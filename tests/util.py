"""Shared helpers for the parity tests (test infrastructure)."""
import functools
import hashlib
import io
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def sha256(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def scene_sha256(s):
    return sha256(np.stack(s.images), s.rot, s.trans, s.feat_pos, *s.feat_refs)


@functools.lru_cache(maxsize=None)
def _rendered_images(name):
    from mve_b200 import synth
    return np.stack(synth.make_scene(name).images)


def golden_scene(name):
    """The scene of fixture `name`.  A fixture whose images would be too large to store holds their SHA-256 instead; they are
    rendered again from the mve_b200.synth config of the same name (rendering is deterministic)."""
    from mve_b200 import synth
    path = os.path.join(GOLD, "%s_scene.npz" % name)
    z = dict(np.load(path))
    if "images" in z:
        return synth.load_scene_npz(path)
    images = _rendered_images(name)
    assert sha256(images) == str(z.pop("images_sha256")), "re-rendered images of %s differ from the fixture's" % name
    buf = io.BytesIO()
    np.savez(buf, images=images, **z)
    buf.seek(0)
    return synth.load_scene_npz(buf)


def golden_ref(name):
    return np.load(os.path.join(GOLD, "%s_ref.npz" % name))


def map_stats(a_depth, b_depth):
    """Fill-mask IoU and relative depth difference percentiles on commonly filled pixels."""
    m1, m2 = a_depth > 0, b_depth > 0
    both = m1 & m2
    iou = both.sum() / max(1, (m1 | m2).sum())
    rel = np.abs(a_depth - b_depth)[both] / a_depth[both]
    return iou, rel, both


def patch_compare(got, ref):
    """Compares PatchOptimization results. Returns dict of mismatch counts / error percentiles."""
    ok_r, ok_g = ref["conf"] > 0, got["conf"] > 0
    both = ok_r & ok_g
    rel = np.abs(got["depth"] - ref["depth"])[both] / np.abs(ref["depth"][both])
    return dict(n=len(ref), ok_mismatch=int((ok_r != ok_g).sum()),
                ids_mismatch=int((got["local_ids"] != ref["local_ids"]).any(-1)[both].sum()),
                rel=rel, conf_abs=np.abs(got["conf"] - ref["conf"])[both],
                dz_abs=np.maximum(np.abs(got["dz_i"] - ref["dz_i"]), np.abs(got["dz_j"] - ref["dz_j"]))[both],
                nrm_abs=np.abs(got["normal"] - ref["normal"]).max(-1)[both], both=both)


def reference_cli_maps(scene, views, threads=None):
    """Runs the UNMODIFIED reference CLI (oracle/_ref/dmrecon, compiled from /root/reference by oracle/Makefile; the
    binary travels to the GPU box) on `scene` for the reference views `views` and returns {view: dict(depth, conf, dz)}.
    One host thread per view like apps/dmrecon/dmrecon.cc:285."""
    import subprocess
    import tempfile
    from mve_b200 import synth
    exe = os.path.join(ROOT, "oracle", "_ref", "dmrecon")
    if not os.path.exists(exe):
        return None
    out = {}
    with tempfile.TemporaryDirectory(prefix="b200mvs_refcli_") as tmp:
        synth.write_mve_scene(scene, tmp)
        cmd = [exe, "-s%d" % scene.scale, "--local-neighbors=%d" % scene.nr_recon_neighbors, "--keep-conf", "--keep-dz",
               "--progress=silent", "--force", "-l" + ",".join(str(v) for v in views), tmp]
        env = dict(os.environ, OMP_NUM_THREADS=str(threads or len(views)))
        r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=3000)
        assert r.returncode == 0, r.stdout + r.stderr
        for v in views:
            vd = os.path.join(tmp, "views", "view_%04d.mve" % v)
            out[v] = dict(depth=synth.read_mvei(os.path.join(vd, "depth-L%d.mvei" % scene.scale))[:, :, 0],
                          conf=synth.read_mvei(os.path.join(vd, "conf-L%d.mvei" % scene.scale))[:, :, 0],
                          dz=synth.read_mvei(os.path.join(vd, "dz-L%d.mvei" % scene.scale)))
    return out


def depthmap_case(kind, seed=0):
    """Inputs of the depth-map consumer tests: (depth, conf) float32 maps."""
    rng = np.random.default_rng(seed)
    if kind == "golden":
        ref = golden_ref("T0")
        return np.ascontiguousarray(ref["depth_0"], np.float32), np.ascontiguousarray(ref["conf_0"], np.float32)
    h, w = (97, 131) if kind == "ragged" else (270, 480)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    d = (5.0 + 0.4 * np.sin(xx / 17.0) + 0.3 * np.cos(yy / 11.0)).astype(np.float32)
    d[(xx > w * 0.6) & (yy > h * 0.3)] += 1.5                      # a depth discontinuity
    hole = rng.random((h, w)) < (0.45 if kind == "ragged" else 0.08)   # ragged: many small islands
    d[hole] = 0.0
    d[:, :3] = 0.0
    conf = rng.random((h, w)).astype(np.float32) - 0.2
    return d, conf


def sampled_maps(name):
    """Stored reference maps of a view too large to store whole: the complete fill mask (`mask`) and depth / conf / dz at a
    seeded sample of its filled pixels (flat indices `idx`)."""
    z = golden_ref(name)
    h, w = z["shape"]
    return dict(mask=np.unpackbits(z["mask"], count=h * w).reshape(h, w).astype(bool), idx=z["idx"], depth=z["depth"],
                conf=z["conf"], dz=z["dz"], scene_sha256=str(z["scene_sha256"]))


def map_parity(ref, got):
    """SURVEY.md 8c map-level figures of `got` against `ref` (dicts with depth, conf, dz).  For a `ref` from sampled_maps the
    fill figures use the complete mask and the error figures the sampled pixels."""
    m_ref = ref["mask"] if "idx" in ref else ref["depth"] > 0
    m_got = got["depth"] > 0
    n_ref = int(m_ref.sum())
    res = dict(iou=float((m_ref & m_got).sum() / max(1, (m_ref | m_got).sum())),
               fill_ratio_diff=float(abs(int(m_got.sum()) - n_ref) / max(1, n_ref)))
    if "idx" in ref:
        got = {k: v.reshape((-1,) + v.shape[2:])[ref["idx"]] for k, v in got.items()}
    _, rel, both = map_stats(ref["depth"], got["depth"])
    res.update(depth_rel_p50=float(np.percentile(rel, 50)), depth_rel_p99=float(np.percentile(rel, 99)),
               depth_rel_le_1e3=float((rel <= 1e-3).mean()), depth_rel_le_1e2=float((rel <= 1e-2).mean()),
               conf_abs_p99=float(np.percentile(np.abs(ref["conf"] - got["conf"])[both], 99)),
               dz_abs_p99=float(np.percentile(np.abs(ref["dz"] - got["dz"])[both].max(-1), 99)), n_both=int(both.sum()))
    if "view_ids" in ref and "view_ids" in got:
        res["view_ids_equal"] = float((ref["view_ids"] == got["view_ids"]).all(-1)[both].mean())
        a, b = ref["view_ids"][both], got["view_ids"][both]
        shared = ((a[:, :, None] == b[:, None, :]) & (a[:, :, None] >= 0)).any(-1).sum(-1)
        res["view_ids_shared_mean"] = float(shared.mean())          # of the (up to) 4 local views of a pixel
        res["view_ids_share_ge3"] = float((shared >= 3).mean())
    return res
