#!/usr/bin/env python
"""bench.py - MVS depth-pixels/second of the dmrecon hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU dmrecon on the host cores
    python bench.py --workload C3|C4|C5 --gpus N ...         # the other BASELINE configs (nominally 8 / 4 / 8 GPUs)
    python bench.py ... --dump-outputs DIR                   # also write the maps of the last timed step (dump_outputs)

Workload (default, N = 1): BASELINE.json configs[1] (C2) - synthetic 16-view 1920x1080 scene, dmrecon scale = 1, all 16
views reconstructed; one step = DMRecon::start for all 16 reference views.  N > 1: the same per-GPU work (16 reference
views per rank, weak scaling) on a 16N-view scene of N tiled camera blocks.  C3 / C4 / C5: the scene is the config's own
(64 / 32 / 128 views); every rank reconstructs views_total / nominal_gpus reference views (8 / 8 / 16), so the config is
covered completely at its nominal GPU count and a shard of it below.  Every rank renders and uploads its own shard; the
images of the other shards arrive through one NCCL all-gather (the reference path has no other cross-view exchange).

value  = depth-pixels (pixels ending with conf > 0, = progress.filled) per second with the image pyramids already
         resident in HBM, results left in HBM, summed over all ranks / max-over-ranks time.
e2e    = the same metric through the public API with HOST buffers: pinned host images -> device (+ all-gather),
         pyramids, reconstruction, depth/conf/dz maps -> pinned host memory, every step.
roofline, cpu_baseline: see DESIGN.md "Measurement".
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "mvs_depth_pixels_per_second"
UNIT = "depth-pixels/s"
VIEWS_PER_GPU = 16


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------------------------------------------
NOMINAL_GPUS = {"C2": 1, "C3": 8, "C4": 4, "C5": 8}


def workload_cfg(name, n_gpus):
    from mve_b200 import synth
    cfg = dict(synth.CONFIGS[name])
    if name == "C2" and n_gpus > 1:
        cfg["views"] = VIEWS_PER_GPU * n_gpus
        cfg["grid"] = (4 * n_gpus, 4)
        cfg["blocks"] = n_gpus            # N copies of the 4x4 camera block side by side; rank r owns block r
        cfg["features"] = 4000 * n_gpus
    cfg["name"] = name
    return cfg


def refs_of_rank(name, cfg, rank, world):
    """Reference views reconstructed by `rank`: C2 - its block of 16; C3/C4/C5 (and test scenes) - a block of
    views_total / nominal_gpus views (the whole config at the nominal GPU count, a shard of it below)."""
    from mve_b200 import sharding
    if name == "C2" or name not in NOMINAL_GPUS:
        return sharding.owned_views(cfg["views"], rank, world)
    per = max(1, cfg["views"] // NOMINAL_GPUS[name])
    lo = min(rank * per, cfg["views"])
    return list(range(lo, min(lo + per, cfg["views"])))


def workload_text(name, scene):
    return "%s: synthetic %d-view %dx%d scene, dmrecon scale=%d" % (name, scene.n_views, scene.width, scene.height, scene.scale)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ----------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own CPU implementation, time-boxed
# ----------------------------------------------------------------------------------------------------------------
def write_scene_for_reference(cfg, views, tmp):
    """Writes the workload as an MVE scene directory (views/*.mve + synth_0.out) for the unmodified reference."""
    from mve_b200 import synth
    s = synth.make_scene(cfg, device="cuda" if _cuda_ok() else None)
    synth.write_mve_scene(s, tmp)
    return s


def _cuda_ok():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


REF_VIEWS_MAX = 16     # the reference arm times a fixed subset of <= 16 reference views (BASELINE.md 4): one thread per view


def run_reference_samples(scene_dir, scene, seconds, views, steps):
    """`steps` bounded samples of the reference CPU path in ONE process. Returns (list of (filled_px, elapsed_s), threads,
    kind, sample_text)."""
    harness = os.path.join(ROOT, "oracle", "_ref", "ref_harness")
    if os.path.exists(harness):
        cmd = [harness, "timed", scene_dir, str(scene.scale), str(scene.nr_recon_neighbors), "%.3f" % seconds, str(steps)] + [str(v) for v in views]
        out = subprocess.run(cmd, capture_output=True, text=True, check=True).stdout.strip().splitlines()
        rows = [json.loads(l) for l in out if l.startswith("{")]
        return [(r["filled"], r["seconds"]) for r in rows], len(views), "reference", \
            "oracle/_ref/ref_harness timed (the unmodified reference, built -O3 -march=x86-64-v3 -funsafe-math-optimizations; " \
            "-march=native is not used because the binary travels): mvs::DMRecon::start of reference views %s on %d host " \
            "threads (one per view, apps/dmrecon.cc:285); clock from the moment every view has reached processQueue " \
            "(RECON_QUEUE) until Progress::cancelled is set %.1f s later; images pre-loaded, pyramids cached" % (
                views, len(views), seconds)
    # the compiled reference is not here: fall back to the CPU port, one thread per view
    from oracle import oracle_py as O
    osc = O.OracleScene(scene)
    st = O.default_settings(scale=scene.scale, nr_recon_neighbors=scene.nr_recon_neighbors)
    rows = []
    for _ in range(steps):
        filled = [0] * len(views)

        def work(k, v):
            filled[k] = int(osc.reconstruct(st, v, max_seconds=seconds)["stats"]["n_filled"])
        t0 = time.time()
        th = [threading.Thread(target=work, args=(k, v)) for k, v in enumerate(views)]
        [t.start() for t in th]
        [t.join() for t in th]
        rows.append((sum(filled), time.time() - t0))
    return rows, len(views), "port", "oracle/mvs_oracle.cc port, %d views on %d threads, stopped after %.1f s" % (len(views), len(views), seconds)


def reference_views(name, cfg, cores):
    """Fixed subset of reference views timed on the CPU: the first block (= the N = 1 workload's views), at most
    REF_VIEWS_MAX and at most one per host core."""
    first = refs_of_rank(name, cfg, 0, max(1, NOMINAL_GPUS.get(name, 1)) if name != "C2" else max(1, cfg.get("blocks", 1)))
    return first[:max(1, min(REF_VIEWS_MAX, cores, len(first)))]


def cpu_baseline_dict(value, threads, kind, sample, cores, n_views):
    return {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample,
            "px_per_s_per_core": value / max(1, threads), "host_cores_available": cores,
            "threads_usable_on_this_workload": min(n_views, cores),
            "note": "the reference's parallelism is one thread per reference view (apps/dmrecon.cc:285); a fixed subset of "
                    "views is timed so that the figure does not depend on the number of GPUs"}


def reference_arm(args, real_stdout):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = workload_cfg(args.workload, max(1, args.gpus))     # the same scene our arm reconstructs at this N
    cores = host_cores()
    n_samples = args.steps + args.warmup
    budget = min(20.0, max(2.0, 150.0 / max(1, n_samples)))
    with tempfile.TemporaryDirectory(prefix="b200mvs_ref_") as tmp:
        t = time.time()
        scene = write_scene_for_reference(cfg, None, tmp)
        views = reference_views(args.workload, cfg, cores)
        log("reference arm: scene written in %.1fs, %d host cores, views %s, %.1fs per step" % (time.time() - t, cores, views, budget))
        rows, threads, kind, sample = run_reference_samples(tmp, scene, budget, views, n_samples)
    for i, (f, el) in enumerate(rows):
        log("  step %d: %d px in %.2fs" % (i, f, el))
    rows = rows[args.warmup:]
    value = sum(f for f, _ in rows) / sum(el for _, el in rows)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(el for _, el in rows) / len(rows), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_text(args.workload, scene),
                       "step": "time-boxed sample of the same workload: %d of its reference views on %d host threads" % (len(views), threads)},
            "cpu_baseline": cpu_baseline_dict(value, threads, kind, sample, cores, scene.n_views),
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), file=real_stdout, flush=True)
    return 0


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
DUMP_BYTES = 60 << 20          # what --dump-outputs writes in all, headers aside


def dump_outputs(path, bufs):
    """Writes the maps a caller of the timed step receives, one row per reference view in order: depth.npy [V, P],
    conf.npy [V, P] and dz.npy [V, P, 2], float32.  P is every pixel of the map, row-major, or, when that would exceed
    DUMP_BYTES, the same sample of pixels in every view: np.sort(np.random.default_rng(0).choice(H * W, P, replace=False)).
    The frontier schedule is not bitwise reproducible at this size, so compare with a tolerance: two runs of the same build
    on C2 (one B200, 1000 W power limit) differed in 0.2-0.7 % of these values, depth by at most 8e-4 relative, with
    identical fill masks."""
    h, w = bufs[0]["depth"].shape
    n = min(h * w, DUMP_BYTES // (16 * len(bufs)))
    idx = np.arange(h * w) if n == h * w else np.sort(np.random.default_rng(0).choice(h * w, n, replace=False))
    os.makedirs(path, exist_ok=True)
    for k, shape in (("depth", (-1,)), ("conf", (-1,)), ("dz", (-1, 2))):
        np.save(os.path.join(path, k + ".npy"), np.stack([b[k].reshape(shape)[idx] for b in bufs]).astype(np.float32))
    log("outputs of the last timed step: %d views x %d of %d pixels -> %s" % (len(bufs), n, h * w, path))


def _protect_stdout():
    """Everything but the one JSON line goes to stderr: libraries (NCCL prints its version banner on stdout) must not
    pollute the line the driver parses.  Returns a file object bound to the original stdout."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    real_stdout = _protect_stdout()
    try:
        return _main(real_stdout)
    finally:
        real_stdout.flush()


def _main(real_stdout):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write depth / conf / dz of the last timed step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(0, args.warmup)
    if args.impl == "reference":
        return reference_arm(args, real_stdout)

    import torch
    import torch.distributed as dist
    from mve_b200 import dmrecon, sharding, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        log("warning: WORLD_SIZE=%d but --gpus %d; using WORLD_SIZE" % (world, args.gpus))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        # one process per GPU on one box: the host phase (b200mvs_plan_views) of every rank starts at the same moment, so
        # each rank takes its share of the cores and leaves the launching threads alone (read by the library per call)
        os.environ.setdefault("B200MVS_HOST_THREADS", str(max(2, (os.cpu_count() or 16) // (2 * world))))

    cfg = workload_cfg(args.workload, world)
    owned = sharding.owned_views(cfg["views"], rank, world)      # views this rank renders / uploads (every view has one owner)
    refs = refs_of_rank(args.workload, cfg, rank, world)          # reference views this rank reconstructs
    t0 = time.time()
    scene = synth.make_scene(cfg, device=str(dev), only_views=owned)
    log("[rank %d] scene %s: %d views (%d owned) generated in %.1fs" % (rank, args.workload, scene.n_views, len(owned), time.time() - t0))
    H, W = scene.height, scene.width

    # pinned host staging of the owned images (the e2e input) and of the result maps (the e2e output)
    host_imgs = torch.empty((len(owned), H, W, 3), dtype=torch.uint8).pin_memory()
    for k, v in enumerate(owned):
        host_imgs[k].copy_(torch.from_numpy(scene.images[v]))
    settings = dmrecon.Settings(scale=scene.scale, nr_recon_neighbors=scene.nr_recon_neighbors)
    gscene = dmrecon.Scene(scene.n_views, device=local)
    gscene.set_features(scene.feat_pos, scene.feat_refs)

    # Cameras of every view are registered once; like the reference (dmrecon.cc:78,238-240) only the images of this rank's
    # reference views and of their selected neighbours are turned into pyramids on this GPU.
    for v in range(scene.n_views):
        gscene.set_view_camera(v, W, H, scene.flen[v], scene.paspect[v], scene.ppoint[v], scene.rot[v], scene.trans[v])
    needed = set(refs)
    for r in refs:
        needed.update(gscene.global_view_selection(settings, r))
    needed = sorted(needed)
    log("[rank %d] %d of %d views needed on this GPU" % (rank, len(needed), scene.n_views))

    exchanged = {"bytes": 0}

    def upload_all():
        """pinned host -> device for the owned views, point-to-point exchange of exactly the images this rank needs from the
        other shards (NCCL over NVLink), pyramids of the needed views."""
        dimgs = host_imgs.to(dev, non_blocking=True)
        imgs, nbytes = sharding.exchange_needed_images(dimgs, owned, needed, scene.n_views, rank, world)
        exchanged["bytes"] = nbytes
        torch.cuda.synchronize()
        for v in needed:
            gscene.set_view_device(v, imgs[v].data_ptr(), W, H, scene.flen[v], scene.paspect[v], scene.ppoint[v],
                                   scene.rot[v], scene.trans[v])
        return imgs

    upload_all()
    Ws, Hs = W, H
    for _ in range(scene.scale):
        Ws, Hs = (Ws + 1) // 2, (Hs + 1) // 2
    out_bufs = []
    for _ in refs:
        out_bufs.append(dict(depth=torch.empty((Hs, Ws), dtype=torch.float32).pin_memory().numpy(),
                             conf=torch.empty((Hs, Ws), dtype=torch.float32).pin_memory().numpy(),
                             dz=torch.empty((Hs, Ws, 2), dtype=torch.float32).pin_memory().numpy()))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # The host part of DMRecon::start (global view selection + seed lists, dmrecon.cc:179-292) of the NEXT step's views is
    # computed on a helper thread while the GPU runs the current step (b200mvs_plan_views) - every step still computes it
    # once, it is just not serialised with the kernel, like consecutive batches of a real scene.
    import concurrent.futures
    planner = concurrent.futures.ThreadPoolExecutor(max_workers=1)
    pending = [planner.submit(gscene.plan_views, settings, refs)]

    plan_wait, call_host = [0.0], [0.0]

    def step_resident(out=None):
        flush.zero_()
        t_w = time.perf_counter()
        pending.pop().result()
        plan_wait[0] += time.perf_counter() - t_w
        pending.append(planner.submit(gscene.plan_views, settings, refs))
        t_c = time.perf_counter()
        _, st = gscene.reconstruct(settings, refs, download=out is not None, out=out)
        call_host[0] += time.perf_counter() - t_c - 1e-3 * st.ms_total_device
        return st

    def step_e2e():
        flush.zero_()
        pending.pop().result()
        upload_all()                                 # re-registers the views: not while the planner reads them
        pending.append(planner.submit(gscene.plan_views, settings, refs))
        _, st = gscene.reconstruct(settings, refs, download=True, out=out_bufs)
        return st

    def agg(x):
        if world == 1:
            return float(x), float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        s = t.clone(); dist.all_reduce(s, op=dist.ReduceOp.SUM)
        m = t.clone(); dist.all_reduce(m, op=dist.ReduceOp.MAX)
        return float(s.item()), float(m.item())

    # ---- HBM-resident timing (value) ----
    for _ in range(args.warmup):
        step_resident()
    barrier()
    stats = []
    plan_wait[0] = call_host[0] = 0.0
    dump = args.dump_outputs and rank == 0
    with ClockSampler(local) as clk:
        t0 = time.perf_counter()
        for i in range(args.steps):
            # the maps stay in HBM, except that the last step of a dumping run copies them to the pinned host buffers
            stats.append(step_resident(out_bufs if dump and i == args.steps - 1 else None))
        barrier()
        elapsed = time.perf_counter() - t0
    clocks = clk.summary()
    if dump:
        dump_outputs(args.dump_outputs, out_bufs)
    filled_local = sum(int(s.n_filled) for s in stats)
    filled_total, _ = agg(filled_local)
    _, elapsed_max = agg(elapsed)
    _, dev_ms_max = agg(sum(s.ms_total_device for s in stats))
    _, plan_wait_max = agg(plan_wait[0])
    _, call_host_max = agg(call_host[0])
    value = filled_total / elapsed_max
    launches_total, _ = agg(sum(int(s.n_kernel_launches) for s in stats))
    refs_total, _ = agg(len(refs))

    # ---- end to end through the host-buffer API ----
    e2e_steps = args.steps
    for _ in range(min(2, args.warmup)):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    f_e2e = 0
    for _ in range(e2e_steps):
        f_e2e += int(step_e2e().n_filled)
    barrier()
    e2e_elapsed = time.perf_counter() - t0
    f_e2e_total, _ = agg(f_e2e)
    _, e2e_max = agg(e2e_elapsed)
    h2d = int(host_imgs.numel())
    d2h = int(sum(b["depth"].nbytes + b["conf"].nbytes + b["dz"].nbytes for b in out_bufs))
    pending.pop().result()
    planner.shutdown()

    # ---- roofline of the dominant kernel (k_frontier: the persistent kernel that runs every PatchOptimization), rank 0 ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    consts = {}
    try:
        consts = json.load(open(os.path.join(ROOT, "profiles", "scene_constants_%s.json" % args.workload)))
    except Exception:
        pass
    bpp = float(consts.get("bytes_alg_per_filled_px", 0.0))
    ms_kernel = sum(s.ms_patch_kernel for s in stats)
    ms_opt = sum(s.ms_optimise_phases for s in stats)
    n_launch = sum(int(s.n_patch_launches) for s in stats)
    achieved = (bpp * filled_local / (ms_kernel * 1e-3)) / 1e9 if ms_kernel > 0 and bpp > 0 else None
    traffic, traffic_src, ncu_context = None, None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_kfrontier_traffic.json")))
        traffic = tj["dram_bytes_per_launch"]
        ncu_context = tj.get("ncu_context")
        traffic_src = tj.get("source")
    except Exception:
        pass
    roofline = {"kernel": "k_frontier (persistent cooperative kernel: seeds + every frontier round of the step in one launch; "
                          "one PatchOptimization per thread in large rounds, per warp in small ones)", "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_filled_px": bpp,
                "definition": "300 B x N_PSE + 75 B x N_opt + 28 B x N_filled with the oracle's strict-order counts per filled "
                              "pixel (profiles/scene_constants_%s.json) x filled pixels of the launch, / CUDA-event time of the "
                              "k_frontier launches in the timed region (one launch per step)" % args.workload,
                "avg_launch_ms": ms_kernel / max(1, n_launch), "launches": n_launch,
                "algorithmic_bytes_per_launch_mean": (bpp * filled_local / max(1, n_launch)) if bpp > 0 else None,
                "kernel_share_of_device_time": ms_kernel / max(1e-9, sum(s.ms_total_device for s in stats)),
                "optimise_phase_share_of_kernel": ms_opt / max(1e-9, ms_kernel),
                "frontier_rounds_per_launch": sum(int(s.n_rounds) for s in stats) / max(1, n_launch),
                "grid_barriers_per_launch": sum(int(s.n_grid_barriers) for s in stats) / max(1, n_launch),
                "impl_sample_sets": sum(int(s.n_sample_sets) for s in stats), "impl_opts": sum(int(s.n_opt) for s in stats),
                "impl_bytes_300_per_set_GBs": (300.0 * sum(int(s.n_sample_sets) for s in stats) / (ms_kernel * 1e-3) / 1e9) if ms_kernel > 0 else None}
    if ncu_context:
        roofline["ncu_context"] = ncu_context      # what actually bounds the kernel, from the committed capture
    # context only: the same launches against the fp32 SIMT peak with SURVEY.md 8(d)'s ~110 kFLOP per reference
    # PatchOptimization (oracle count per filled pixel x filled pixels)
    opf = float(consts.get("opt_per_filled_px", 0.0))
    if ms_kernel > 0 and opf > 0:
        tf = 110e3 * opf * filled_local / (ms_kernel * 1e-3) / 1e12
        roofline["fp32_context"] = {"achieved_tflops": tf, "peak_tflops": 74.0, "frac": tf / 74.0,
                                    "note": "148 SM x 128 lanes x 2 x 1.965 GHz (derived, not measured); 110 kFLOP per reference optimisation"}

    # ---- cpu_baseline (rank 0): the reference's own CPU dmrecon on this box's host cores, bounded sample ----
    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        try:
            full = synth.make_scene(cfg, device=str(dev))
            with tempfile.TemporaryDirectory(prefix="b200mvs_cpu_") as tmp:
                synth.write_mve_scene(full, tmp)
                cores = host_cores()
                views = reference_views(args.workload, cfg, cores)
                rows, threads, kind, sample = run_reference_samples(tmp, full, args.cpu_seconds / 3.0, views, 3)
            rows = rows[1:]                      # the first sample builds the reference's lazy pyramid levels
            cpu_baseline = cpu_baseline_dict(sum(f for f, _ in rows) / sum(el for _, el in rows), threads, kind, sample, cores, full.n_views)
        except Exception as ex:   # the GPU numbers stand on their own
            cpu_baseline = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": repr(ex)}
    if world > 1:
        barrier()

    # ---- sub-line: the consumer of the maps (SURVEY 8f rank 2), depthmap_triangulate of one result map on the device ----
    depthmap_ops = None
    if rank == 0:
        try:
            from mve_b200 import depthmap as D
            dmap = np.ascontiguousarray(out_bufs[0]["depth"])
            ax = float(max(Ws, Hs))
            invproj = np.array([1 / ax, 0, -0.5 * Ws / ax, 0, 1 / ax, -0.5 * Hs / ax, 0, 0, 1], np.float32)
            D.depthmap_triangulate(dmap, invproj, device=local)
            tri = D.depthmap_triangulate(dmap, invproj, device=local)
            nv, nf = len(tri["vertices"]), len(tri["faces"])
            # algorithmic bytes: depth in (4 B/px), vertex ids out (4 B/px), vertices 12 B, faces 12 B each
            alg = dmap.size * 8 + nv * 12 + nf * 12
            depthmap_ops = {"op": "depthmap_triangulate (libs/mve/depthmap.cc:196-375) of one %dx%d result map" % (Ws, Hs),
                            "device_ms": tri["device_ms"], "vertices": nv, "faces": nf,
                            "algorithmic_GBs": alg / (tri["device_ms"] * 1e-3) / 1e9 if tri["device_ms"] > 0 else None,
                            "note": "kernels + one scan, device time; a map of this size is launch-latency bound"}
        except Exception as ex:
            depthmap_ops = {"error": repr(ex)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * elapsed_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_text(args.workload, scene),
                           "reference_views_per_gpu": len(refs), "reference_views_total": int(refs_total),
                           "sharding": ("reference views block-sharded over ranks; each rank receives exactly the neighbour images it needs from their owners "
                                        "(NCCL send/recv, %.0f MB per step on rank 0)" % (exchanged["bytes"] / 1e6)) if world > 1 else "single GPU",
                           "l2": "256 MiB buffer written between steps (L2 flush); the pyramids alone (%.0f MB incl. quad texels) exceed the 126 MB L2" %
                                 (len(needed) * W * H * 20 * 4 / 3 / 1e6),
                           "host_phase": "global view selection + seed lists of step k+1 are computed on a helper thread while the GPU runs step k (b200mvs_plan_views)",
                           "filled_px_per_step": filled_total / args.steps, "swept_px_per_step": int(refs_total) * Ws * Hs,
                           "device_ms_per_step_max": dev_ms_max / args.steps,
                           "host_phase_wait_ms_per_step_max": 1e3 * plan_wait_max / args.steps,
                           "call_minus_kernel_ms_per_step_max": 1e3 * call_host_max / args.steps},
                "clocks": clocks, "gpu_launches": int(launches_total),
                "e2e": {"value": f_e2e_total / e2e_max, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "steps": e2e_steps, "ms_per_step": 1e3 * e2e_max / e2e_steps},
                "roofline": roofline, "cpu_baseline": cpu_baseline, "depthmap_ops": depthmap_ops}
        print(json.dumps(line), file=real_stdout, flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
