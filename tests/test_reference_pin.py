"""Pins the CPU oracle against the REFERENCE ITSELF: the reference's gpu_process.cu compiled unmodified
(oracle/build_ref.py, stand-in Eigen header) and run on a B200, its outputs recorded with the inputs they came
from in tests/golden/reference_pin_v1.npz (tests/golden/make_reference_pin.py).

  * -fmad=false build: every output the oracle restates must be bit-identical
    (map_index, height, variance, transformed x/y, fused elevation/variance/colour, scroll state);
  * reference's own flags (FMA contraction on): cell indices identical except where a point
    sits within float rounding of a cell edge, heights/variances within 1e-5 relative
    (BASELINE.json north_star tolerance);
  * features / ray clean-up use CUDA's libm trig in the reference and the deterministic trig in
    the oracle: compared with a tolerance and a bounded mismatch fraction.
The reference's `lowest` update is a data race (gpu_process.cu:434-438); it is compared only
where a cell received a single point."""
import os
import sys

import numpy as np
import pytest

import gem_b200
from gem_b200 import synth
from oracle_lib import OracleMap

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_reference_pin as pin  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", pin.NAME)


@pytest.fixture(scope="module")
def ref():
    g = np.load(GOLD, allow_pickle=False)
    assert "reference gpu_process.cu" in str(g["generated_by"])
    return g


def bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


def _inputs(g, prefix):
    return {"xyzi": g[prefix + "xyzi"], "rgba": g[prefix + "rgba"], "T": g[prefix + "T"], "position": g[prefix + "pos"]}


def _frame(fr, **kw):
    return gem_b200.make_frame(fr["T"], gem_b200.LaserSensorProcessor(), **kw)


def test_process_points_and_fuse_bit_exact_vs_reference_nofma(ref):
    fr = _inputs(ref, "pp_in_")   # reference demo axes: the reference hard-codes the box filter (gpu_process.cu:393)
    L, res = 200, 0.1
    o = OracleMap(L, res, compat_box_filter=True)
    f = _frame(fr)
    cr, co = [ref["pp_" + n] for n in ("centre", "start", "shift")], o.move(fr["position"])
    for a, b in zip(cr, co):
        assert np.array_equal(a, b)
    x, y, z = (fr["xyzi"][:, k] for k in range(3))
    kr = [ref["pp_" + n] for n in ("key", "var", "xt", "yt", "zt")]
    ko = o.process_points(x, y, z, f)
    for a, b, name in zip(kr, ko, ["map_index", "var", "x_ts", "y_ts", "z_ts"]):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), name
    assert (kr[0] >= 0).sum() > 5000
    # lowest: race-free where a cell got exactly one point
    key = kr[0]
    geo = np.array([o.points_to_index(a, b)[0] for a, b in zip(kr[2][key >= 0], kr[3][key >= 0])])
    u, c = np.unique(geo, return_counts=True)
    single = u[c == 1]
    lr, lo = ref["pp_lowest"].reshape(-1), o.get_layer("lowest").reshape(-1)
    assert np.array_equal(bits(lr[single]), bits(lo[single])) and single.size > 500
    R, G, B = (fr["rgba"][:, k].astype(np.int32) for k in range(3))
    for rep in range(2):
        o.fuse_points(key, R, G, B, fr["xyzi"][:, 3], kr[4], kr[1])
    fo = o.map_feature()
    for name in ("elevation", "variance", "intensity", "color_r", "color_g", "color_b"):
        assert np.array_equal(ref["pp_feat_" + name].view(np.uint32), fo[name].view(np.uint32)), name


def test_dense_collisions_order_is_index_order_in_the_reference(ref):
    """G_fuse visits a cell's points in ascending index: the O(N) oracle must agree on a cloud
    with hundreds of points per cell (gates, replacements, floors)."""
    L, res = 48, 0.25
    c = pin.dense_cloud()        # behind the sensor so the hard-coded box filter keeps the points
    assert pin.digest(c["xyzi"], c["rgba"]) == str(ref["dense_sha256"]), "not the cloud the reference was run on"
    T = synth.pose_matrix(0.0, pin.DENSE_SHIFT_Y, 0.5, 0.0)
    f = gem_b200.make_frame(T, gem_b200.LaserSensorProcessor(ignore_points_above=5, ignore_points_below=-5))
    o = OracleMap(L, res, compat_box_filter=True)
    x, y, z = (c["xyzi"][:, k] for k in range(3))
    kr0 = ref["dense_key"].astype(np.int32)
    ko = o.process_points(x, y, z, f)
    assert np.array_equal(kr0, ko[0]) and (kr0 >= 0).sum() > 20000
    R, G, B = (c["rgba"][:, k].astype(np.int32) for k in range(3))
    o.fuse_points(ko[0], R, G, B, c["xyzi"][:, 3], ko[4], ko[1])
    fo = o.map_feature()
    for name in ("elevation", "variance", "intensity", "color_r"):
        assert np.array_equal(ref["dense_feat_" + name].view(np.uint32), fo[name].view(np.uint32)), name


def test_stream_with_scroll_features_and_raytracing_vs_reference(ref):
    L, res = 160, 0.1
    o = OracleMap(L, res, compat_box_filter=True)
    worst_trav, cleaned_r, cleaned_o, ray_mismatch, valid_total = 0.0, 0, 0, 0, 0
    for k in range(5):
        p = f"strm{k}_"
        fr = _inputs(ref, p + "in_")
        f = _frame(fr)
        cr, co = [ref[p + n] for n in ("centre", "start", "shift")], o.move(fr["position"])
        for a, b in zip(cr, co):
            assert np.array_equal(a, b), "Move outputs"
        x, y, z = (fr["xyzi"][:, j] for j in range(3))
        ko = o.process_points(x, y, z, f)
        assert np.array_equal(ref[p + "key"], ko[0])
        R, G, B = (fr["rgba"][:, j].astype(np.int32) for j in range(3))
        o.fuse_points(ko[0], R, G, B, fr["xyzi"][:, 3], ko[4], ko[1])
        # the reference's racy lowest differs from the oracle's definition where several points
        # share a cell: it was given the oracle's lowest layer before the ray step
        fr_ = {n: ref[p + "feat_" + n] for n in ("elevation", "variance", "traver")}
        fo = o.map_feature()
        assert np.array_equal(bits(fr_["elevation"]), bits(fo["elevation"])), f"frame {k} elevation"
        assert np.array_equal(bits(fr_["variance"]), bits(fo["variance"])), f"frame {k} variance"
        valid = fo["elevation"] != -10
        both = valid & (fo["traver"] != -10)
        assert np.array_equal(fr_["traver"][valid] == -10, fo["traver"][valid] == -10)
        d = np.abs(fr_["traver"][both] - fo["traver"][both])
        d = d[~np.isnan(d)]
        # CUDA libm trig vs the deterministic trig: tiny differences, rare Jacobi-iteration flips
        assert np.mean(d < 1e-4) > 0.995, float(np.mean(d < 1e-4))
        worst_trav = max(worst_trav, float(np.percentile(d, 99.9)) if d.size else 0.0)
        # the ray step was made comparable: the reference was given the oracle's traver layer
        er0 = ref[p + "elev_before_ray"]
        o.raytracing()
        er, eo = ref[p + "elev_after_ray"], o.get_layer("elevation")
        cleaned_r += int(((er == -10) & (er0 != -10)).sum())
        cleaned_o += int(((eo == -10) & (er0 != -10)).sum())
        ray_mismatch += int((bits(er) != bits(eo)).sum())
        valid_total += int(valid.sum())
        o.set_layer("elevation", er)   # keep the two in lock step for the next frame
    assert cleaned_r > 0 and ray_mismatch == 0, (cleaned_r, cleaned_o, ray_mismatch)
    assert worst_trav < 5e-2


def test_reference_with_fma_contraction_within_tolerance(ref):
    """the reference's own build flags (no -fmad=false): indices identical away from cell edges,
    heights / variances within 1e-5 relative of the oracle"""
    fr = _inputs(ref, "fma_in_")
    L, res = 200, 0.1
    o = OracleMap(L, res, compat_box_filter=True)
    f = _frame(fr)
    o.move(fr["position"])
    x, y, z = (fr["xyzi"][:, k] for k in range(3))
    kr = {1: ref["fma_var"], 4: ref["fma_zt"], 0: ref["fma_key"]}
    ko = o.process_points(x, y, z, f)
    acc = (kr[0] >= 0) | (ko[0] >= 0)
    diff = kr[0] != ko[0]
    assert diff.sum() <= max(3, int(2e-4 * acc.sum())), int(diff.sum())   # only points on a cell edge
    same = ~diff & (ko[0] >= 0)
    for a, b in ((kr[1], ko[1]), (kr[4], ko[4])):
        assert np.allclose(a[same], b[same], rtol=1e-5, atol=0)
    R, G, B = (fr["rgba"][:, k].astype(np.int32) for k in range(3))
    o.fuse_points(ko[0], R, G, B, fr["xyzi"][:, 3], ko[4], ko[1])
    fr_, fo = {n: ref["fma_feat_" + n] for n in ("elevation", "variance")}, o.map_feature()
    valid = fo["elevation"] != -10
    close_e = np.isclose(fr_["elevation"][valid], fo["elevation"][valid], rtol=1e-5, atol=1e-7)
    close_v = np.isclose(fr_["variance"][valid], fo["variance"][valid], rtol=1e-5, atol=0)
    # a gate decision can flip when |dh|/sigma is within rounding of 5: bounded fraction
    assert close_e.mean() > 0.9995 and close_v.mean() > 0.9995, (close_e.mean(), close_v.mean())
