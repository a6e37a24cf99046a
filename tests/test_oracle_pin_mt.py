"""Pins the multi-frame restatement (oracle/sf_oracle_mt.cpp) and the restated third-party pieces.

  * tests/golden/mt_*.npz: outputs of the reference's UNMODIFIED Variational_MT driver (oracle/_ref, built against
    header shims) -- bit for bit, both SOR orderings, occlusion labels and the returned average change included.
  * oracle/_ref itself when present: more configurations, bit for bit.
  * cv::GaussianBlur / cv::resize restatement vs python cv2 (only where cv2 is importable: the build container).
  * the binary min-cut (gco stand-in) vs brute force.
"""
import ctypes as C
import itertools
import os

import numpy as np
import pytest

import mt_helpers as mh
from golden.make_golden_mt import CASES

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("name", sorted(CASES))
def test_mt_restatement_matches_golden(oracle, name):
    c = CASES[name]
    g = np.load(os.path.join(GOLD, name + ".npz"))
    ims, wx, wy = mh.window(c["size"][0], c["size"][1], c["S"], zero_flow=c.get("zero", False))
    p = mh.params(c["S"], **c["kw"])
    for mode, tag in ((0, "lex"), (1, "rb")):
        r = mh.run_cpu(oracle.lib, "sfo_", ims, wx, wy, p, mode)
        assert np.array_equal(r["wx"].array, g["wx_" + tag]) and np.array_equal(r["wy"].array, g["wy_" + tag]), (name, tag)
        assert np.array_equal(r["occ"].array, g["occ_" + tag])
        assert np.array_equal(np.array(r["avg"], np.float32), g["avg_" + tag])
    assert np.array_equal(np.array([r["params"].img_norm_avg[k] for k in range(3)], np.float32), g["norm_avg"])
    assert np.array_equal(np.array([r["params"].img_norm_std[k] for k in range(3)], np.float32), g["norm_std"])


@pytest.mark.parametrize("S,kw", [
    (3, dict()),
    (2, dict(robust_color=4, robust_color_eps=0.5, dataterm=0, occlusion_reasoning=0)),
    (4, dict(one_direction=1, rho=[1, 1, 1], omega=[0, 2, 1], smoothing=0, robust_grad=2, robust_grad_eps=0.5)),
])
def test_mt_operator_entries_compose_to_one_iteration(oracle, S, kw):
    """sfo_mt_system -> sfo_sor_coupled -> wx + du is exactly sfo_variational_mt with one alternation, one outer and one inner
    iteration: the operator entries are the functions the pinned driver is made of."""
    from slowflow_b200 import ColorImage, Image
    w, h = 61, 45
    ims, wx, wy = mh.window(w, h, S)
    p = mh.params(S, niter_alter=1, niter_outer=1, niter_inner=1, **kw)
    rng = np.random.default_rng(3)
    chw = ColorImage.from_array(rng.uniform(0.5, 1.5, size=(3, h, w)).astype(np.float32))
    full = mh.run_cpu(oracle.lib, "sfo_", ims, wx, wy, p, 1, chw)
    frames = [f.copy() for f in ims]
    q = mh.clone_params(p)
    oracle.lib.sfo_normalize(mh.frame_array(frames), len(frames), C.byref(q))
    occ = Image(w, h)
    occ.buf[:] = -1.0 if (p.occlusion_reasoning or p.one_direction) else 0.0
    A = [Image(w, h) for _ in range(7)]
    assert oracle.lib.sfo_mt_system(*[a.ptr() for a in A], mh.frame_array(frames), wx.ptr(), wy.ptr(), None, None, occ.ptr(),
                                    chw.ptr(), C.byref(q)) == 0
    du, dv = Image(w, h), Image(w, h)
    oracle.lib.sfo_sor_coupled(du.ptr(), dv.ptr(), *[a.ptr() for a in A], q.niter_solver, q.sor_omega, 1)
    assert np.array_equal(wx.array + du.array, full["wx"].array)
    assert np.array_equal(wy.array + dv.array, full["wy"].array)
    assert np.abs(du.array).max() > 1e-3


@pytest.mark.parametrize("size,S,kw", [
    ((131, 77), 3, dict(niter_alter=2, niter_outer=2, robust_color=4, robust_color_eps=0.5)),
    ((96, 64), 3, dict(niter_alter=1, niter_outer=1, robust_color=3, robust_color_truncation=5.0, dataterm=0)),
    ((128, 96), 4, dict(niter_alter=1, niter_outer=2, one_direction=1, rho=[1, 1, 1], omega=[0, 2, 1])),
    ((160, 120), 2, dict(niter_alter=3, niter_outer=10, thres_outer=5e-3, occlusion_reasoning=0)),
    ((120, 90), 3, dict(niter_alter=2, niter_outer=2, graphcut_int_terms=1, robust_grad=2, robust_grad_eps=0.5)),
    ((150, 100), 3, dict(layers=3, niter_alter=1, niter_outer=2, smoothing=0, robust_reg=2, robust_reg_eps=0.5)),
])
def test_mt_restatement_bit_identical_to_reference_driver(oracle, reference, size, S, kw):
    ims, wx, wy = mh.window(size[0], size[1], S)
    p = mh.params(S, **kw)
    for mode in (0, 1):
        a = mh.run_cpu(reference.lib, "sf_ref_", ims, wx, wy, p, mode)
        b = mh.run_cpu(oracle.lib, "sfo_", ims, wx, wy, p, mode)
        assert np.array_equal(a["wx"].array, b["wx"].array) and np.array_equal(a["wy"].array, b["wy"].array)
        assert np.array_equal(a["occ"].array, b["occ"].array) and a["avg"] == b["avg"]
        assert a["stats"][1] == b["stats"][1]  # graph-cut calls
        for x, y in zip(a["frames"], b["frames"]):
            assert np.array_equal(x.array, y.array)  # normalize()


def test_blur_resize_restatement_matches_cv2(reference):
    cv2 = pytest.importorskip("cv2")
    L = reference.lib
    FP = C.POINTER(C.c_float)
    L.sf_ref_blur_resize.argtypes = [FP, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, FP]
    r = np.random.RandomState(0)
    img = (r.rand(97, 131, 3) * 255).astype(np.float32)
    sigma = 1 / np.sqrt(2 * 0.9)
    for dr, dc, sg in [(97, 131, sigma), (87, 117, 0.0), (87, 117, sigma), (150, 200, 0.0)]:
        out = np.zeros((dr, dc, 3), np.float32)
        L.sf_ref_blur_resize(img.ctypes.data_as(FP), 97, 131, 3, sg, dr, dc, out.ctypes.data_as(FP))
        ref = img
        if sg > 0:
            ref = cv2.GaussianBlur(ref, (0, 0), sg, sigmaY=sg, borderType=cv2.BORDER_REPLICATE)
        if (dr, dc) != (97, 131):
            ref = cv2.resize(ref, (dc, dr), interpolation=cv2.INTER_LINEAR)
        assert np.abs(out - ref).max() <= 1e-5 * 255  # cv2 4.13: blur within 2e-7, resize within 5e-6 (relative to 255)


def test_mincut_standin_is_optimal(reference):
    L = reference.lib
    FP = C.POINTER(C.c_float)
    L.sf_ref_mincut.argtypes = [C.c_int, C.c_int, FP, FP, C.c_float, C.c_int, C.POINTER(C.c_int)]
    r = np.random.RandomState(1)
    w, h = 4, 3
    q = lambda v: np.round(np.asarray(v, np.float64) * 2 ** 24) / 2 ** 24

    def energy(lab, d0, d1, a):
        e = sum(d1[p] if lab[p] else d0[p] for p in range(w * h))
        for y in range(h):
            for x in range(w):
                p = y * w + x
                e += a * (int(x + 1 < w and lab[p] != lab[p + 1]) + int(y + 1 < h and lab[p] != lab[p + w]))
        return e

    for _ in range(60):
        d0, d1, a = r.rand(w * h).astype(np.float32), r.rand(w * h).astype(np.float32), np.float32(r.rand() * 0.5)
        lab = np.zeros(w * h, np.int32)
        L.sf_ref_mincut(w, h, d0.ctypes.data_as(FP), d1.ctypes.data_as(FP), a, 0, lab.ctypes.data_as(C.POINTER(C.c_int)))
        best = min(energy(l, q(d0), q(d1), float(q(a))) for l in itertools.product([0, 1], repeat=w * h))
        assert abs(energy(lab, q(d0), q(d1), float(q(a))) - best) < 1e-9
    # integer EnergyTermType: every cost < 1 truncates to 0 -> nothing leaves label 0
    lab = np.ones(w * h, np.int32)
    L.sf_ref_mincut(w, h, d0.ctypes.data_as(FP), d1.ctypes.data_as(FP), a, 1, lab.ctypes.data_as(C.POINTER(C.c_int)))
    assert not lab.any()


def test_prescale_restatement_matches_cv2(oracle):
    """slow_flow.cpp:538-542 on a CV_32F image: GaussianBlur(Size(), s, s, BORDER_REPLICATE) + resize(Size(0,0), f, f,
    INTER_LINEAR).  The resize-by-factor form rounds the size (cvRound) and maps coordinates with 1/f."""
    cv2 = pytest.importorskip("cv2")
    from slowflow_b200 import ColorImage
    from slowflow_b200.image import color_image_t
    L = oracle.lib
    CP = C.POINTER(color_image_t)
    L.sfo_prescale.argtypes = [CP, CP, C.c_float]
    L.sfo_prescale_size.argtypes = [C.c_int, C.c_int, C.c_float, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    r = np.random.RandomState(5)
    for (w, h, f) in [(131, 97, 0.5), (200, 150, 0.75), (97, 61, 0.9), (64, 48, 0.3), (80, 60, 1.5)]:
        img = (r.rand(h, w, 3) * 255).astype(np.float32)
        sg = 1 / np.sqrt(np.float64(np.float32(2 * f)))
        ref = cv2.GaussianBlur(img, (0, 0), sg, sigmaY=sg, borderType=cv2.BORDER_REPLICATE)
        ref = cv2.resize(ref, None, fx=float(np.float32(f)), fy=float(np.float32(f)), interpolation=cv2.INTER_LINEAR)
        ow, oh = C.c_int(), C.c_int()
        assert L.sfo_prescale_size(w, h, f, C.byref(ow), C.byref(oh)) == 0
        assert (oh.value, ow.value) == ref.shape[:2]
        src = ColorImage.from_array(np.ascontiguousarray(img.transpose(2, 0, 1)))
        dst = ColorImage(ow.value, oh.value)
        assert L.sfo_prescale(dst.ptr(), src.ptr(), f) == 0
        assert np.abs(dst.array - ref.transpose(2, 0, 1)).max() <= 1e-5 * 255
