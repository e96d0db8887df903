"""Pins the C port (oracle/stereo_oracle.c) to the reference's OWN compiled code: oracle/_ref is the reference's
src/{CVC,CVF,DispSel}.cpp built unmodified against oracle/shim (only the five OpenCV image primitives are stand-ins,
themselves pinned against cv2 in test_oracle.py).  What that library returned on the inputs below is stored in
tests/golden/golden_ref.{json,npz} (tests/golden/make_golden_ref.py), so the port is held to it on every machine:
_ref == port == golden."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, read_png


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def golden_ref():
    with open(os.path.join(GOLDEN, "golden_ref.json")) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def golden_ref_arrays():
    return np.load(os.path.join(GOLDEN, "golden_ref.npz"))


@pytest.mark.parametrize("scene", ["Cones", "Teddy"])
def test_ref_equals_port_equals_golden(scene, oracle_scene_results, golden, golden_ref):
    port = oracle_scene_results[scene]
    ref = golden_ref["scenes"][scene]
    for k_ref, k_port in (("lGrd", "lg"), ("rGrd", "rg"), ("lRaw", "lraw"), ("rRaw", "rraw"),
                          ("lVol", "lf"), ("rVol", "rf"), ("lDis", "ld"), ("rDis", "rd")):
        assert sha(port[k_port]) == ref[k_ref], f"{scene}: reference {k_ref} != port {k_port}"
    s = scene.lower()
    assert ref["lDis"] == sha(read_png(os.path.join(GOLDEN, f"{s}_lDis.png")))
    assert ref["rDis"] == sha(read_png(os.path.join(GOLDEN, f"{s}_rDis.png")))
    # the cv2-driven golden hashes (tests/golden/make_golden.py) hold for the reference's compiled code as well
    g = golden["scenes"][scene]
    for gk, rk in (("lGrd", "lGrd"), ("rGrd", "rGrd"), ("lRaw", "lRaw"), ("rRaw", "rRaw"),
                   ("lFilt", "lVol"), ("rFilt", "rVol"), ("lDis", "lDis"), ("rDis", "rDis")):
        assert ref[rk] == g[gk], f"{scene}: reference {rk} differs from the cv2-driven golden hash"


def test_ref_thread_counts_and_both_code_paths(scenes, oracle, golden_ref):
    """threads = 1, 3, 8 (remainder batches, DispEst.cpp:238) give the same volumes in the reference and in the port;
    the reference's non-pthread twins buildCV_left/right (CVC.cpp:122-179) and CVSelect_thread (DispSel.cpp:53-81)
    agree with the pthread / OpenMP variants, and so with the port."""
    _, _, l, r = scenes["Teddy"]
    l, r = l[:60, :128].copy(), r[:60, :128].copy()
    D = 12
    ref = golden_ref["threads"]
    keys = ("lRaw", "rRaw", "lVol", "rVol", "lDis", "rDis")
    for t in ("1", "3"):
        for k in keys:
            assert ref[t][k] == ref["8"][k], (t, k)
    for t in (1, 3, 8):
        _, _, lraw, rraw = oracle.cost_const(l, r, D, threads=t)
        port = oracle.pipeline(l, r, D, threads=t, keep_volumes=True)
        got = dict(lRaw=lraw, rRaw=rraw, lVol=port["lVol"], rVol=port["rVol"], lDis=port["lDis"], rDis=port["rDis"])
        for k in keys:
            assert sha(got[k]) == ref[str(t)][k], (t, k)
    for d in (0, 5, 11):
        assert golden_ref["buildcv"][f"left_d{d}"] == sha(lraw[d])
        assert golden_ref["buildcv"][f"right_d{d}"] == sha(rraw[d])
    assert golden_ref["wta"]["thread_variant_4"] == ref["8"]["lDis"]
    assert golden_ref["wta"]["pthread_8"] == sha(oracle.wta(port["lVol"]))


def test_ref_guided_filter_on_arbitrary_costs(oracle, golden_ref_arrays):
    """GuidedFilter_cv compiled from the reference vs the port on signed, wide-range caller-provided costs."""
    z = golden_ref_arrays
    img = z["gf_img"]
    rgb, mean, var = oracle.cvf_preprocess(img)
    for k in range(3):                      # cost scales 1, 1e-4, 300
        assert np.array_equal(oracle.guided_filter(rgb, mean, var, z[f"gf_p{k}"]), z[f"gf_q{k}"]), k


def test_ref_gray_mode_switch(scenes, oracle, golden_ref):
    _, _, l, r = scenes["Cones"]
    l, r = l[:40, :90].copy(), r[:40, :90].copy()
    for gm in (0, 1):
        ref = golden_ref["gray_mode"][str(gm)]
        lg, rg, lraw, rraw = oracle.cost_const(l, r, 6, gray_mode=gm)
        assert sha(lg) == ref["lGrd"] and sha(lraw) == ref["lRaw"] and sha(rraw) == ref["rRaw"], gm
