"""Golden vectors of the reference's OWN compiled operators -- TEST INFRASTRUCTURE.

oracle/_ref/libstereo_ref.so is PRiMEStereoMatch's src/{CVC,CVF,DispSel}.cpp and include/JointWMF.h compiled
unmodified against oracle/shim (recipe: `make -C oracle ref REF=<PRiMEStereoMatch checkout>`).  The checkout is not
part of this repository, so this script runs that library once on the inputs of tests/test_oracle_ref.py and of the
reference-JointWMF tests in tests/test_pp.py and stores what it returned; the tests then hold the C port
(oracle/stereo_oracle.c) to these outputs on every machine.

Writes
  tests/golden/golden_ref.json     sha256 of the reference's outputs (scene volumes, thread counts, code paths, gray modes,
                                   post-processed maps of the posterised images) and the number of distinct 6-bit colours
                                   of each posterised feature image
  tests/golden/golden_ref.npz      the reference's guided filter on seeded random costs (inputs and outputs) and its
                                   post-processed map (u8) of the natural Teddy left image with its colour count
Run: python tests/golden/make_golden_ref.py"""
import hashlib
import json
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import oracle as O  # noqa: E402
from oracle import ref as R  # noqa: E402


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def posterise(img8, masks=(0xE0, 0xE0, 0xC0)):
    return (img8 & np.array(masks, np.uint8)).astype(np.uint8)


def scene(name):
    s = name.lower()
    l8 = cv2.imread(os.path.join(HERE, f"{s}_im2.png"), cv2.IMREAD_UNCHANGED)
    r8 = cv2.imread(os.path.join(HERE, f"{s}_im6.png"), cv2.IMREAD_UNCHANGED)
    return l8, r8, O.u8_to_f32(l8), O.u8_to_f32(r8)


def main():
    if not R.available():
        raise SystemExit(f"{R.PATH} is not built: `make -C oracle ref REF=<PRiMEStereoMatch checkout>`")
    js = {"generator": "tests/golden/make_golden_ref.py", "scenes": {}}
    arrays = {}

    # whole CVC -> CVF -> WTA path on both Middlebury scenes, D = 64
    full = {}
    for name in ("Cones", "Teddy"):
        l8, r8, l, r = scene(name)
        res = R.pipeline(l, r, 64, threads=8, keep=True)
        full[name] = res
        js["scenes"][name] = {k: sha(res[k]) for k in ("lGrd", "rGrd", "lRaw", "rRaw", "lVol", "rVol", "lDis", "rDis")}

    # thread counts (remainder batches) and the non-pthread twins of buildCV / CVSelect, Teddy crop, D = 12
    _, _, l, r = scene("Teddy")
    l, r = l[:60, :128].copy(), r[:60, :128].copy()
    threads = {}
    for t in (1, 3, 8):
        res = R.pipeline(l, r, 12, threads=t, keep=True)
        threads[str(t)] = {k: sha(res[k]) for k in ("lRaw", "rRaw", "lVol", "rVol", "lDis", "rDis")}
        if t == 8:
            base = res
    js["threads"] = threads
    js["buildcv"] = {f"{side}_d{d}": sha(R.buildcv(l, r, d, right=(side == "right")))
                     for side in ("left", "right") for d in (0, 5, 11)}
    js["wta"] = {"thread_variant_4": sha(R.wta(base["lVol"], thread_variant=True, threads=4)),
                 "pthread_8": sha(R.wta(base["lVol"]))}

    # gray-mode switch of the cost construction, Cones crop, D = 6
    _, _, l, r = scene("Cones")
    l, r = l[:40, :90].copy(), r[:40, :90].copy()
    js["gray_mode"] = {}
    for gm in (0, 1):
        res = R.pipeline(l, r, 6, gray_mode=gm, keep=True)
        js["gray_mode"][str(gm)] = {k: sha(res[k]) for k in ("lGrd", "lRaw", "rRaw")}

    # GuidedFilter_cv on signed, wide-range caller-provided costs
    rng = np.random.default_rng(8)
    H, W = 48, 77
    img = rng.random((H, W, 3), dtype=np.float32)
    arrays["gf_img"] = img
    for k, scale in enumerate((1.0, 1e-4, 300.0)):
        p = (rng.normal(0, 1, (H, W)) * scale).astype(np.float32)
        arrays[f"gf_p{k}"] = p
        arrays[f"gf_q{k}"] = R.guided_filter(img, p)

    # PP::processDM through the reference's JointWMF: posterised images (<= 256 colours, clustering exact) on both
    # views of both scenes, and the natural Teddy left image (> 256 colours, clustered by the shim's k-means)
    js["post_process_posterised"] = {}
    for name in ("Cones", "Teddy"):
        l8, r8, _, _ = scene(name)
        for view, img8, dk in (("l", l8, "lDis"), ("r", r8, "rDis")):
            want, ncol = R.post_process(O.u8_to_f32(posterise(img8)), full[name][dk])
            js["post_process_posterised"][f"{name}_{view}"] = {"sha256": sha(want), "ncol": ncol}
    _, _, l, _ = scene("Teddy")
    want, ncol = R.post_process(l, full["Teddy"]["lDis"])
    arrays["pp_teddy_l_natural"] = want
    arrays["pp_teddy_l_natural_ncol"] = np.int32(ncol)

    with open(os.path.join(HERE, "golden_ref.json"), "w") as f:
        json.dump(js, f, indent=1)
        f.write("\n")
    np.savez_compressed(os.path.join(HERE, "golden_ref.npz"), **arrays)


if __name__ == "__main__":
    main()
