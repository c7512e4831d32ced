"""Mints the committed golden fixtures from the REFERENCE ITSELF (oracle/_ref, built by oracle/Makefile from the
reference tree).  Needs that tree and oracle/_ref:   python tests/golden/make_golden.py [fixture ...]   (default: all)

Outputs (all under tests/golden/):
  srgb2lin.npy            the 256-entry table of libs/dmrecon/mvs_tools.cc:30-95, parsed from the source
  <S>_scene.npz           the synthetic scene (images, cameras, features) so that fixtures are self-contained; images over
                          1 MB are stored as their SHA-256 and rendered again by tests/util.golden_scene
  <S>_ref.npz             reference results for that scene:
      gvs_default / gvs_n3     "Global View Selection:" line of the reference per view (default and -n 3)
      patch_in / patch_out     inputs and mvs::PatchOptimization results through oracle/_ref/ref_harness
      depth_v / conf_v / dz_v  maps written by oracle/_ref/dmrecon for views v (apps/dmrecon CLI, unmodified)
      undist_v                 pyramid level `scale` written by the reference (scale != 0 only)
  T0_seed77_ref.npz       patch_in / patch_out on a scene no other fixture uses (only its SHA-256 is stored)
  C2_view5_ref.npz,       one view of BASELINE-size scenes through oracle/_ref/dmrecon: the complete fill mask and
  C5r_view3_ref.npz       depth / conf / dz at a seeded sample of the filled pixels (tests/util.sampled_maps)
  dmops_ref.npz           libs/mve/depthmap.cc through `ref_harness dmops` on the inputs of tests/test_gpu_depthmap_ops.py:
                          SHA-256 of every exact output, a seeded sample of the vertices for the float ones
"""
import os
import re
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from mve_b200 import synth            # noqa: E402
from oracle import oracle_py as O     # noqa: E402
from tests.util import depthmap_case, golden_scene, reference_cli_maps, scene_sha256, sha256   # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
REF = os.path.join(ROOT, "oracle", "_ref")


def parse_lut():
    src = open("/root/reference/libs/dmrecon/mvs_tools.cc").read()
    a = src.index("srgb2lin[256] = {")
    body = src[a:src.index("};", a)]
    vals = [np.float32(x.rstrip("f")) for x in re.findall(r"[0-9.]+(?:e-?[0-9]+)?f", body)]
    assert len(vals) == 256
    return np.asarray(vals, np.float32)


def run_cli(scene_dir, scale, nrn, extra=()):
    cmd = [os.path.join(REF, "dmrecon"), "-s%d" % scale, "--local-neighbors=%d" % nrn, "--keep-conf", "--keep-dz",
           "--progress=silent", "--force"] + list(extra) + [scene_dir]
    return subprocess.run(cmd, capture_output=True, text=True, check=True, env=dict(os.environ, OMP_NUM_THREADS="1")).stdout


def gvs_lines(scene_dir, scale, nrn, n_views, extra=()):
    out = {}
    for v in range(n_views):
        txt = subprocess.run([os.path.join(REF, "dmrecon"), "-s%d" % scale, "--local-neighbors=%d" % nrn,
                              "--progress=simple", "--force", "-l%d" % v] + list(extra) + [scene_dir],
                             capture_output=True, text=True).stdout
        m = re.search(r"Global View Selection:([ 0-9]*)", txt)
        out[v] = np.asarray([int(x) for x in m.group(1).split()], np.int32) if m else np.zeros(0, np.int32)
    return out


def save_scene(s, name):
    path = os.path.join(GOLD, "%s_scene.npz" % name)
    synth.save_scene_npz(s, path)
    images = np.stack(s.images)
    if images.nbytes > 1 << 20:
        z = dict(np.load(path))
        del z["images"]
        np.savez_compressed(path, images_sha256=sha256(images), **z)
    return golden_scene(name)


def mint_gvs_only(name):
    """Only the printed global view selections (many-candidate scene)."""
    s = save_scene(synth.make_scene(name), name)
    tmp = tempfile.mkdtemp(prefix="golden_")
    try:
        synth.write_mve_scene(s, tmp)
        data = {}
        for tag, extra in (("gvs_default", ()), ("gvs_n3", ("-n3",))):
            for v, ids in gvs_lines(tmp, s.scale, s.nr_recon_neighbors, s.n_views, extra).items():
                data["%s_%d" % (tag, v)] = ids
        np.savez_compressed(os.path.join(GOLD, "%s_ref.npz" % name), **data)
        print(name, "gvs only;", "view 0 ->", data["gvs_default_0"])
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def mint(name, map_views, n_patches=1500):
    s = save_scene(synth.make_scene(name), name)
    tmp = tempfile.mkdtemp(prefix="golden_")
    try:
        synth.write_mve_scene(s, tmp)
        data = {}
        for tag, extra in (("gvs_default", ()), ("gvs_n3", ("-n3",))):
            g = gvs_lines(tmp, s.scale, s.nr_recon_neighbors, s.n_views, extra)
            for v, ids in g.items():
                data["%s_%d" % (tag, v)] = ids
        run_cli(tmp, s.scale, s.nr_recon_neighbors)
        for v in map_views:
            vd = os.path.join(tmp, "views", "view_%04d.mve" % v)
            data["depth_%d" % v] = synth.read_mvei(os.path.join(vd, "depth-L%d.mvei" % s.scale))[:, :, 0]
            data["conf_%d" % v] = synth.read_mvei(os.path.join(vd, "conf-L%d.mvei" % s.scale))[:, :, 0]
            data["dz_%d" % v] = synth.read_mvei(os.path.join(vd, "dz-L%d.mvei" % s.scale))
            if s.scale:
                data["undist_%d" % v] = synth.read_mvei(os.path.join(vd, "undist-L%d.png" % s.scale))
        # patch-level vectors: realistic inputs = a slice of the oracle's own execution trace (seeds + queue)
        osc = O.OracleScene(s)
        st = O.default_settings(scale=s.scale, nr_recon_neighbors=s.nr_recon_neighbors)
        ref = map_views[0]
        r = osc.reconstruct(st, ref, trace_cap=200000)
        tin = r["trace_in"]
        seeds = np.nonzero(tin["n_local"] == 0)[0]
        rest = np.nonzero(tin["n_local"] != 0)[0]
        rng = np.random.default_rng(7)
        pick = np.sort(np.concatenate([seeds, rng.choice(rest, size=min(n_patches, len(rest)), replace=False)]))
        pin = np.ascontiguousarray(tin[pick])
        # a few hostile inputs: image border, negative depth slope, far-off depth
        extra = np.zeros(6, O.PATCH_IN)
        extra["local_ids"] = -1
        extra[0] = (1, 1, 5.0, 0, 0, 0, [-1] * 4)
        extra[1] = (s.width // (2 ** s.scale) - 2, 10, 5.0, 0, 0, 0, [-1] * 4)
        extra[2] = (40, 40, 5.0, -3.0, 0.0, 0, [-1] * 4)
        extra[3] = (40, 40, 50.0, 0, 0, 0, [-1] * 4)
        extra[4] = (40, 40, 0.5, 0, 0, 0, [-1] * 4)
        extra[5] = (40, 40, -1.0, 0, 0, 0, [-1] * 4)
        pin = np.concatenate([pin, extra])
        data["patch_gvs"], data["patch_out"] = harness_patches(s, tmp, ref, pin)
        data["patch_ref_view"] = np.int32(ref)
        data["patch_in"] = pin
        np.savez_compressed(os.path.join(GOLD, "%s_ref.npz" % name), **data)
        print(name, "patches", len(pin), "maps", map_views)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def harness_patches(s, scene_dir, ref, pin):
    """mvs::PatchOptimization of the reference on the inputs `pin` (ref_harness patches): (global view selection, results)."""
    fin, fout = os.path.join(scene_dir, "pin.bin"), os.path.join(scene_dir, "pout.bin")
    pin.tofile(fin)
    txt = subprocess.run([os.path.join(REF, "ref_harness"), "patches", scene_dir, str(ref), str(s.scale),
                          str(s.nr_recon_neighbors), fin, fout], capture_output=True, text=True, check=True).stdout
    m = re.search(r"Global View Selection:([ 0-9]*)", txt)
    return np.asarray([int(x) for x in m.group(1).split()], np.int32), np.fromfile(fout, dtype=O.PATCH_OUT)


def mint_fresh_patches():
    """The first 3000 optimisations of the restatement's strict-order run of view 1 on a T0-like scene with another seed."""
    s = synth.make_scene("T0", seed=77, features=200)
    st = O.default_settings(scale=s.scale, nr_recon_neighbors=s.nr_recon_neighbors)
    pin = O.OracleScene(s).reconstruct(st, 1, trace_cap=3000)["trace_in"]
    tmp = tempfile.mkdtemp(prefix="golden_")
    try:
        synth.write_mve_scene(s, tmp)
        gvs, pout = harness_patches(s, tmp, 1, pin)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    np.savez_compressed(os.path.join(GOLD, "T0_seed77_ref.npz"), scene_sha256=scene_sha256(s), patch_gvs=gvs, patch_in=pin,
                        patch_out=pout)


def mint_sampled_maps(name, s, view, n=4096):
    ref = reference_cli_maps(s, [view])[view]
    mask = ref["depth"] > 0
    idx = np.sort(np.random.default_rng(0).choice(np.flatnonzero(mask), n, replace=False)).astype(np.uint32)
    np.savez_compressed(os.path.join(GOLD, "%s_ref.npz" % name), scene_sha256=scene_sha256(s),
                        shape=np.asarray(mask.shape), mask=np.packbits(mask), idx=idx, depth=ref["depth"].reshape(-1)[idx],
                        conf=ref["conf"].reshape(-1)[idx], dz=ref["dz"].reshape(-1, 2)[idx])
    print(name, "filled", int(mask.sum()))


def mint_dmops(n=512):
    data = {}
    with tempfile.TemporaryDirectory(prefix="golden_") as tmp:
        def harness(*args):
            subprocess.run([os.path.join(REF, "ref_harness"), "dmops"] + [str(a) for a in args], check=True)

        def load(path, dtype=np.float32):
            return np.fromfile(os.path.join(tmp, path), dtype)
        for kind in ("golden", "ragged", "large"):
            dm, cm = depthmap_case(kind)
            h, w = dm.shape
            dm.tofile(os.path.join(tmp, "dm.f32"))
            cm.tofile(os.path.join(tmp, "cm.f32"))
            harness("confclean", w, h, os.path.join(tmp, "dm.f32"), os.path.join(tmp, "cm.f32"), os.path.join(tmp, "cc.f32"))
            data["%s_confclean" % kind] = sha256(load("cc.f32"))
            for thres in (1, 7, 50, 2000):
                harness("cleanup", w, h, thres, os.path.join(tmp, "dm.f32"), os.path.join(tmp, "cl.f32"))
                data["%s_cleanup_%d" % (kind, thres)] = sha256(load("cl.f32"))
        for kind, dd, color in (("golden", 5.0, True), ("ragged", 5.0, False), ("large", 0.0, True), ("large", 2.0, False)):
            dm, _ = depthmap_case(kind, seed=3)
            h, w = dm.shape
            ax = float(max(w, h))
            invproj = np.array([1 / ax, 0, -0.5 * w / ax, 0, 1 / ax, -0.5 * h / ax, 0, 0, 1], np.float32)
            dm.tofile(os.path.join(tmp, "dm.f32"))
            cpath = "-"
            if color:
                cpath = os.path.join(tmp, "ci.u8")
                np.random.default_rng(1).integers(0, 255, size=(h, w, 3), dtype=np.uint8).tofile(cpath)
            harness("triangulate", w, h, repr(dd), os.path.join(tmp, "dm.f32"), cpath, 3, *[repr(float(v)) for v in invproj],
                    os.path.join(tmp, "out"))
            key = "%s_%g_%d_" % (kind, dd, color)
            verts = load("out.verts").reshape(-1, 3)
            idx = np.sort(np.random.default_rng(0).choice(len(verts), min(n, len(verts)), replace=False))
            data[key + "n_vertices"] = len(verts)
            data[key + "idx"] = idx.astype(np.uint32)
            data[key + "vertices"] = verts[idx]
            if color:
                data[key + "colors"] = load("out.colors").reshape(-1, 4)[idx]
            data[key + "normals"] = load("out.normals").reshape(-1, 3)[idx]
            data[key + "scales"] = load("out.scales")[idx]
            data[key + "vertex_ids"] = sha256(load("out.vids", np.uint32))
            data[key + "faces"] = sha256(load("out.faces", np.uint32))
            data[key + "n_faces"] = len(load("out.faces", np.uint32)) // 3
            data[key + "confidences"] = sha256(load("out.confs"))
    np.savez_compressed(os.path.join(GOLD, "dmops_ref.npz"), **data)


FIXTURES = {
    "srgb": lambda: np.save(os.path.join(GOLD, "srgb2lin.npy"), parse_lut()),
    "T0": lambda: mint("T0", [0, 3]),
    "T1": lambda: mint("T1", [4]),
    "T2": lambda: mint("T2", [0]),
    "T4": lambda: mint("T4", [1]),
    "T3": lambda: mint_gvs_only("T3"),
    "T0_seed77": mint_fresh_patches,
    "C2_view5": lambda: mint_sampled_maps("C2_view5", synth.make_scene("C2"), 5),
    "C5r_view3": lambda: mint_sampled_maps("C5r_view3", synth.make_scene("C5", views=32, width=640, height=480, features=6000,
                                                                         orbit_views_per_ring=16), 3, n=2048),
    "dmops": mint_dmops,
}

if __name__ == "__main__":
    for f in sys.argv[1:] or FIXTURES:
        FIXTURES[f]()
