#!/usr/bin/env python
"""Generate the committed golden fixture tests/golden/gem_golden_v1.npz.

Inputs: a seeded 3-frame HDL-64E-shaped stream (subsampled to keep the file small), reference
demo axes (so the hard-coded box filter of gpu_process.cu:393 keeps points), 96x96 @ 0.2 m map.
Outputs per frame, produced by THE REFERENCE ITSELF when run where oracle/_ref exists and a GPU
is present: Move outputs, Process_points outputs, and the layers after Fuse / Map_feature /
Raytracing, from
  ref_nofma : the reference's gpu_process.cu compiled unmodified with -fmad=false
  ref_fma   : the same file with the reference's own flags (FMA contraction on)
plus the CPU oracle's traversability / roughness / slope on the same inputs (its other outputs are
bit-identical to ref_nofma's and are not stored twice).  Only what tests/test_golden.py reads is
kept, LZMA-compressed, so that the file stays under 1 MB.

  python tests/golden/make_golden.py [OUTDIR]      # needs a GPU and oracle/_ref; default tests/golden
"""
import io
import os
import sys
import zipfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import gem_b200  # noqa: E402
from gem_b200 import synth  # noqa: E402
from oracle_lib import OracleMap  # noqa: E402

L, RES, NFRAMES, STRIDE = 96, 0.2, 3, 11
EXACT = ("key", "var", "xt", "yt", "zt", "centre", "start", "shift", "feat_elevation", "feat_variance", "feat_intensity",
         "feat_color_r", "feat_color_g", "feat_color_b", "elev_after_ray")
STORED = {"ref_nofma": EXACT + ("feat_traver",), "ref_fma": ("key", "zt", "var", "feat_elevation"),
          "oracle": ("feat_traver", "feat_rough", "feat_slope")}


def savez_lzma(path, arrays):
    """np.savez with LZMA-compressed members (np.load reads them like any .npz)"""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_LZMA) as z:
        for name in sorted(arrays):
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(arrays[name]), allow_pickle=False)
            z.writestr(name + ".npy", buf.getvalue())


def stored(tag, res):
    return {f"{tag}_{k}": v for k, v in res.items() if k.split("_", 1)[1] in STORED[tag]}


def inputs():
    scene = synth.make_scene()
    out = []
    for k in range(NFRAMES):
        fr = synth.hdl64_frame(k, scene=scene, compat_axes=True, speed=8.0)
        fr["xyzi"] = np.ascontiguousarray(fr["xyzi"][k::STRIDE])
        fr["rgba"] = np.ascontiguousarray(fr["rgba"][k::STRIDE])
        fr["rgba"][::13, 1] = 0          # exercise the "any channel zero -> keep old colour" rule
        out.append(fr)
    return out


def run(m, frames, is_ref, lowest_from=None):
    """drive one implementation; returns dict of arrays"""
    res = {}
    for k, fr in enumerate(frames):
        f = gem_b200.make_frame(fr["T"], gem_b200.LaserSensorProcessor())
        centre, start, shift = m.move(fr["position"])
        x, y, z = (fr["xyzi"][:, j] for j in range(3))
        key, var, xt, yt, zt = m.process_points(x, y, z, f)
        R, G, B = (fr["rgba"][:, j].astype(np.int32) for j in range(3))
        m.fuse_points(key, R, G, B, fr["xyzi"][:, 3], zt, var)
        if is_ref and lowest_from is not None:
            # the reference's `lowest` update is a data race; use the oracle's definition so the
            # ray step is comparable (documented in tests/test_reference_pin.py)
            m.set_layer("lowest", lowest_from[k])
        feat = m.map_feature()
        m.raytracing()
        res[f"f{k}_centre"], res[f"f{k}_start"], res[f"f{k}_shift"] = centre, start, shift
        res[f"f{k}_key"], res[f"f{k}_var"], res[f"f{k}_xt"], res[f"f{k}_yt"], res[f"f{k}_zt"] = key, var, xt, yt, zt
        for name in ("elevation", "variance", "intensity", "color_r", "color_g", "color_b", "rough", "slope", "traver"):
            res[f"f{k}_feat_{name}"] = feat[name]
        res[f"f{k}_elev_after_ray"] = m.get_layer("elevation").reshape(-1)
    return res


def main():
    import torch
    import ref_lib
    if not (torch.cuda.is_available() and ref_lib.available(True) and ref_lib.available(False)):
        sys.exit("needs a GPU and both reference builds in oracle/_ref (python oracle/build_ref.py)")
    frames = inputs()
    data = {"L": L, "res": RES, "nframes": NFRAMES}
    for k, fr in enumerate(frames):
        data[f"in{k}_xyzi"], data[f"in{k}_rgba"], data[f"in{k}_T"], data[f"in{k}_pos"] = fr["xyzi"], fr["rgba"], fr["T"], fr["position"]
    # oracle (also records its lowest layer after process_points for the reference's ray step)
    o = OracleMap(L, RES, compat_box_filter=True)
    lows = []

    class Spy:
        def __getattr__(self, n):
            return getattr(o, n)

        def fuse_points(self, *a):
            lows.append(o.get_layer("lowest").copy())
            return o.fuse_points(*a)
    data.update(stored("oracle", run(Spy(), frames, False)))
    for tag, nofma in (("ref_nofma", True), ("ref_fma", False)):
        r = ref_lib.RefMap(L, RES, nofma=nofma)
        data.update(stored(tag, run(r, frames, True, lowest_from=lows)))
    data["generated_by"] = "reference gpu_process.cu on " + torch.cuda.get_device_name(0)
    outdir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    os.makedirs(outdir, exist_ok=True)
    path = os.path.join(outdir, "gem_golden_v1.npz")
    savez_lzma(path, data)
    print("wrote", path, os.path.getsize(path), "bytes;", data["generated_by"])


if __name__ == "__main__":
    main()
