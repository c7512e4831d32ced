"""Map-level parity at BASELINE size (-m gpu): one full view of C2 (1920x1080, scale 1) and one view of a reduced C5 orbit
scene, GPU vs the UNMODIFIED reference CLI (oracle/_ref/dmrecon, strict priority order) on the same scene (stored by
tests/golden/make_golden.py as the complete fill mask and depth / conf / dz at a seeded sample of the filled pixels).
Tolerances: SURVEY.md 8c map level - fill-mask IoU >= 0.98, fill ratio within 1 %, depth rel. err <= 1e-3 on >= 99 % and
<= 1e-2 on >= 99.9 % of the commonly filled pixels, dz abs err p99 <= 5e-3; the confidence figure depends on WHICH seed's
region claims a pixel (the local view set is inherited from the parent), i.e. on the processing order: asserted per mode at
the measured level (DESIGN.md "Frontier schedule" has the table)."""
import pytest

from tests.util import map_parity, sampled_maps, scene_sha256

pytestmark = pytest.mark.gpu


def test_C2_full_view_vs_reference_cli():
    from mve_b200 import dmrecon, synth
    s = synth.make_scene("C2", device="cuda")
    view = 5
    ref = sampled_maps("C2_view5")
    assert scene_sha256(s) == ref["scene_sha256"], "the scene differs from the one the reference ran on"
    g = dmrecon.Scene.from_synth(s)
    res = {}
    for mode, kw in [("default", {}), ("topk_256", dict(frontier_topk=256)), ("topk_64", dict(frontier_topk=64))]:
        maps, st = g.reconstruct(dmrecon.Settings(scale=s.scale, **kw), [view])
        r = map_parity(ref, maps[0])
        r["rounds"], r["n_opt"], r["device_ms"] = int(st.n_rounds), int(st.n_opt), float(st.ms_total_device)
        res[mode] = r
    for mode, r in res.items():
        assert r["iou"] >= 0.98 and r["fill_ratio_diff"] <= 0.01, (mode, r)
        assert r["depth_rel_le_1e3"] >= 0.99 and r["depth_rel_le_1e2"] >= 0.999, (mode, r)
        assert r["dz_abs_p99"] <= 5e-3, (mode, r)
    assert res["default"]["conf_abs_p99"] <= 4e-2, res["default"]
    assert res["topk_256"]["conf_abs_p99"] <= 1.5e-2, res["topk_256"]
    assert res["topk_256"]["conf_abs_p99"] < res["default"]["conf_abs_p99"]
    # frontier_topk = 64 meets every map-level figure of SURVEY 8c, the confidence bound included
    assert res["topk_64"]["conf_abs_p99"] <= 5e-3, res["topk_64"]


def test_C5_reduced_orbit_view_vs_reference_cli():
    """C5 geometry (two-ring orbit around the blob) with 32 views of 640x480: the poorly conditioned case (grazing views,
    ~35 % fill).  The reference differs from ITSELF here at this level when only the order of equal-priority pops changes
    (oracle strict vs reference CLI: tests/test_oracle_vs_reference.py), so the depth bound is the measured one."""
    from mve_b200 import dmrecon, synth
    s = synth.make_scene("C5", device="cuda", views=32, width=640, height=480, features=6000, orbit_views_per_ring=16)
    view = 3
    ref = sampled_maps("C5r_view3")
    assert scene_sha256(s) == ref["scene_sha256"], "the scene differs from the one the reference ran on"
    g = dmrecon.Scene.from_synth(s)
    maps, st = g.reconstruct(dmrecon.Settings(scale=s.scale), [view])
    r = map_parity(ref, maps[0])
    assert r["iou"] >= 0.95, r
    assert r["depth_rel_le_1e2"] >= 0.99, r
    assert r["depth_rel_p50"] <= 5e-4, r
