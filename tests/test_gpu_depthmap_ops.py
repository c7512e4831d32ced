"""Depth-map consumers on the device (-m gpu) against the REFERENCE's own functions (libs/mve/depthmap.cc) run through
oracle/_ref/ref_harness dmops on the same buffers (tests/golden/dmops_ref.npz, minted by tests/golden/make_golden.py):
depthmap_confidence_clean, depthmap_cleanup (bit-exact) and depthmap_triangulate - vertex ids, faces and vertex count exact,
vertices / colours exact up to the reference binary's own -funsafe-math contraction (<= 1e-6 relative).  Exact outputs are
compared through their SHA-256, float outputs at a seeded sample of the vertices."""
import numpy as np
import pytest

from tests.util import depthmap_case, golden_ref, sha256

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("kind", ["golden", "ragged", "large"])
def test_confidence_clean_and_cleanup_bit_exact(kind):
    from mve_b200 import depthmap as D
    ref = golden_ref("dmops")
    dm, cm = depthmap_case(kind)
    got = dm.copy()
    D.depthmap_confidence_clean(got, cm)
    assert sha256(got) == str(ref["%s_confclean" % kind])
    for thres in (1, 7, 50, 2000):
        got = D.depthmap_cleanup(dm, thres)
        assert sha256(got) == str(ref["%s_cleanup_%d" % (kind, thres)]), thres
    # empty and full maps
    z = np.zeros((5, 7), np.float32)
    assert (D.depthmap_cleanup(z, 3) == 0).all()
    o = np.ones((5, 7), np.float32)
    assert (D.depthmap_cleanup(o, 35) == 1).all() and (D.depthmap_cleanup(o, 36) == 0).all()


@pytest.mark.parametrize("kind,dd,color", [("golden", 5.0, True), ("ragged", 5.0, False), ("large", 0.0, True), ("large", 2.0, False)])
def test_triangulate_matches_reference(kind, dd, color):
    from mve_b200 import depthmap as D
    z = golden_ref("dmops")
    key = "%s_%g_%d_" % (kind, dd, color)
    idx = z[key + "idx"].astype(np.int64)
    verts, nrm, scl = z[key + "vertices"], z[key + "normals"], z[key + "scales"]
    dm, _ = depthmap_case(kind, seed=3)
    h, w = dm.shape
    ax = float(max(w, h))
    invproj = np.array([1 / ax, 0, -0.5 * w / ax, 0, 1 / ax, -0.5 * h / ax, 0, 0, 1], np.float32)
    ci = None
    if color:
        ci = np.random.default_rng(1).integers(0, 255, size=(h, w, 3), dtype=np.uint8)
    got = D.depthmap_triangulate(dm, invproj, dd_factor=dd, color=ci)
    assert int(z[key + "n_vertices"]) > 100 and int(z[key + "n_faces"]) > 100
    # the rest of scene2pset's per-view work: vertex normals (angle-weighted), boundary confidences (exact: ring / 4), scale values
    ps = D.depthmap_pointset(dm, invproj, dd_factor=dd, color=ci, with_normals=True, conf_iterations=4, scale_factor=2.5)
    assert sha256(ps["faces"]) == str(z[key + "faces"])
    assert sha256(ps["vertex_ids"]) == str(z[key + "vertex_ids"])
    cfs = ps["confidences"]
    assert sha256(cfs) == str(z[key + "confidences"])
    assert set(np.unique(cfs)).issubset({0.0, 0.25, 0.5, 0.75, 1.0}) and (cfs == 0).any()
    assert kind == "ragged" or (cfs == 1).any()        # a ragged map may have no vertex further than 4 rings from a boundary
    dn = np.abs(ps["normals"][idx] - nrm).max(-1)
    # angle weights are acos() of float dot products (device acosf vs the host's libm): measured p99.9 3.4e-5, max 6.7e-5
    assert np.percentile(dn, 99.9) <= 1e-4 and dn.max() <= 2e-3, (np.percentile(dn, 99.9), dn.max())
    ds = np.abs(ps["scales"][idx] - scl) / np.abs(scl).max()
    assert ds.max() <= 3e-5, ds.max()          # float sums over <= 9 neighbours, the reference binary contracts to FMAs
    assert sha256(got["vertex_ids"]) == str(z[key + "vertex_ids"])
    assert got["faces"].shape == (int(z[key + "n_faces"]), 3) and sha256(got["faces"]) == str(z[key + "faces"])
    assert got["vertices"].shape == (int(z[key + "n_vertices"]), 3)
    assert np.abs(got["vertices"][idx] - verts).max() <= 1e-6 * np.abs(verts).max()
    if color:
        assert np.abs(got["colors"][idx] - z[key + "colors"]).max() <= 1e-6
    # world transform = the reference's mesh_transform of the same vertices
    ctw = np.eye(4, dtype=np.float32)
    ctw[:3, :3] = np.array([[0.36, 0.48, -0.8], [-0.8, 0.6, 0.0], [0.48, 0.64, 0.6]], np.float32)
    ctw[:3, 3] = [1.5, -2.0, 0.25]
    gw = D.depthmap_triangulate(dm, invproj, dd_factor=dd, cam_to_world=ctw)
    want = verts @ ctw[:3, :3].T + ctw[:3, 3]
    assert np.abs(gw["vertices"][idx] - want).max() <= 2e-6 * np.abs(want).max()
    assert sha256(gw["faces"]) == str(z[key + "faces"])
