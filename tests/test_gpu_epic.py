"""EPIC sparse-to-dense interpolation on the GPU (slowflow_b200/csrc/sf_epic.cu, SURVEY 8f rank 4) against the reference's
own unmodified epic.cpp / epic_aux.cpp compiled into oracle/_ref (LAPACK's sgels_ comes from oracle/ref_glue/lapack_stub.c:
parity unpinned at that one call).

Synthetic matches and edge costs (slowflow_b200.synth.epic_case): the real inputs -- DeepMatching matches, SED edges -- are
not available offline.  The discrete parts are compared exactly: the label map of the geodesic distance transform, the k
nearest seeds and their distances, the surviving matches.  The dense flow is gated like every other flow on this path:
mean endpoint difference <= 0.01 px, max <= 0.1 px."""
import ctypes as C

import numpy as np
import pytest

import epic_helpers as eh
from epic_helpers import epic_inputs, nnfield_inputs
from slowflow_b200 import ColorImage, Image, synth
from slowflow_b200.api import EpicParams, epic_params_default
from slowflow_b200.image import color_image_t, image_t

pytestmark = pytest.mark.gpu


def ref_lib(reference):
    L = reference.lib
    IP, CP = C.POINTER(image_t), C.POINTER(color_image_t)
    L.sf_ref_epic.argtypes = [IP, IP, CP, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(EpicParams)]
    L.sf_ref_epic.restype = None
    L.sf_ref_dist_trf_nnfield.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int]
    L.sf_ref_dist_trf_nnfield.restype = None
    return L


@pytest.mark.parametrize("w,h,ns,nn,kind", [
    (97, 61, 40, 10, "texture"), (200, 150, 300, 26, "texture"), (64, 64, 64, 26, "flat"), (333, 211, 900, 100, "texture"),
    (1024, 436, 5000, 100, "texture"), (130, 33, 50, 50, "ridges"),
    # geometry of the strip pipeline: narrower than a 32-column block, five rows, exactly / just over the 96-column window of a
    # strip row, a last strip of one row; zero cost (the square root of the update at its argument 0)
    (31, 7, 12, 5, "texture"), (100, 5, 9, 4, "texture"), (96, 32, 30, 10, "texture"), (97, 33, 30, 10, "ridges"), (70, 50, 25, 8, "zero"),
])
def test_nnfield_labels_and_neighbours_equal_reference(ctx, reference, w, h, ns, nn, kind):
    """dist_trf_nnfield_subset (epic_aux.cpp:350-401): the sweeps are reproduced operation for operation, so the label map
    is identical; the neighbour lists are identical including the order among equal distances (same heap discipline)."""
    L = ref_lib(reference)
    seeds, cost = nnfield_inputs(w, h, ns, kind)
    rb, rd, rl = np.zeros((ns, nn), np.int32), np.zeros((ns, nn), np.float32), np.zeros((h, w), np.int32)
    c2 = cost.copy()
    L.sf_ref_dist_trf_nnfield(rb.ctypes.data, rd.ctypes.data, rl.ctypes.data, seeds.ctypes.data, ns, nn, c2.ctypes.data, w, h)
    gl, gb, gd, sweeps = ctx.epic_nnfield(seeds, nn, cost)
    print("%dx%d %s: %d seeds, %d sweeps" % (w, h, kind, ns, sweeps))
    assert np.array_equal(gl, rl), "labels differ at %d pixels" % int((gl != rl).sum())
    assert np.array_equal(gb, rb), "neighbour lists differ in %d entries" % int((gb != rb).sum())
    assert np.array_equal(gd, rd)


@pytest.mark.parametrize("w,h,n,method", [(320, 200, 800, "LA"), (320, 200, 800, "NW"), (1024, 436, 5000, "LA"), (501, 333, 2500, "LA")])
def test_epic_matches_reference(ctx, reference, w, h, n, method):
    L = ref_lib(reference)
    im, m, edges = synth.epic_case(w, h, n)
    ci = ColorImage.from_array(im)
    p = epic_params_default()
    p.method = method.encode()
    rx, ry = Image(w, h), Image(w, h)
    e_ref = edges.copy()
    L.sf_ref_epic(rx.ptr(), ry.ptr(), ci.ptr(), m.ctypes.data, n, 4, e_ref.ctypes.data, C.byref(p))
    gx, gy = Image(w, h), Image(w, h)
    e_gpu = edges.copy()
    st = ctx.epic(gx, gy, ci, m, e_gpu, p)
    assert np.array_equal(e_gpu, e_ref)  # += euc in the caller's array, like the reference
    assert st.matches_in == n and 0 < st.matches_after_consistency < n  # the outliers are filtered
    d = np.sqrt((gx.array - rx.array) ** 2 + (gy.array - ry.array) ** 2)
    u, v = synth.gt_flow(w, h)
    print("%dx%d %s: %d -> %d -> %d matches, sweeps %d/%d, GPU vs reference mean %.3e max %.3e px; EPE vs GT %.3f"
          % (w, h, method, st.matches_in, st.matches_after_saliency, st.matches_after_consistency, st.sweeps_prefilter,
             st.sweeps_interpolation, d.mean(), d.max(), float(np.sqrt((gx.array - u) ** 2 + (gy.array - v) ** 2).mean())))
    assert d.mean() <= 0.01 and d.max() <= 0.1


def test_epic_filters_off_and_few_matches(ctx, reference):
    """saliency_th = pref_nn = 0 (both filters off), fewer matches than nn (nns = number of matches, epic.cpp:185)."""
    L = ref_lib(reference)
    w, h, n = 160, 120, 37
    im, m, edges = synth.epic_case(w, h, n, outliers=0.0)
    ci = ColorImage.from_array(im)
    p = epic_params_default()
    p.saliency_th, p.pref_nn = 0.0, 0
    rx, ry, gx, gy = Image(w, h), Image(w, h), Image(w, h), Image(w, h)
    e_ref, e_gpu = edges.copy(), edges.copy()  # (named: a temporary would be freed before the call reads it)
    L.sf_ref_epic(rx.ptr(), ry.ptr(), ci.ptr(), m.ctypes.data, n, 4, e_ref.ctypes.data, C.byref(p))
    st = ctx.epic(gx, gy, ci, m, e_gpu, p)
    assert st.matches_after_consistency == n
    d = np.sqrt((gx.array - rx.array) ** 2 + (gy.array - ry.array) ** 2)
    assert d.mean() <= 0.01 and d.max() <= 0.1


def test_epic_then_variational_pipeline(ctx):
    """The two steps of epicflow.cpp:125-127 back to back on the device path: interpolate, then refine."""
    w, h = 320, 200
    im, m, edges = synth.epic_case(w, h, 900)
    f0, f1 = ColorImage.from_array(synth.frame(w, h, 0)), ColorImage.from_array(synth.frame(w, h, 1))
    wx, wy = Image(w, h), Image(w, h)
    ctx.epic(wx, wy, f0, m, edges, None)
    u, v = synth.gt_flow(w, h)
    before = float(np.sqrt((wx.array - u) ** 2 + (wy.array - v) ** 2)[8:-8, 8:-8].mean())
    ctx.variational(wx, wy, f0, f1, None)
    after = float(np.sqrt((wx.array - u) ** 2 + (wy.array - v) ** 2)[8:-8, 8:-8].mean())
    print("EPE vs GT: interpolated %.3f -> refined %.3f" % (before, after))
    # (the synthetic ground truth is only approximate at the motion discontinuity, SURVEY 8d: no strict improvement is
    # guaranteed there; the refinement must keep the interpolated field's quality and stay finite)
    assert np.isfinite(wx.array).all() and after < 1.25 * before and after < 0.5



# Regression vectors (tests/golden/make_golden_epic.py): the GPU path's own outputs on the cases above, recorded when they
# were added.  They are NOT the reference's outputs and do not replace the comparisons above; they make a change of the EPIC
# kernels' results visible where the reference build is absent.  Discrete parts must stay equal; the dense flow may move by a tenth of the reference gate
# (mean 0.001 px, max 0.01 px), so that the recorded vectors cannot take up more than that of the reference tolerance.
@pytest.mark.parametrize("w,h,ns,nn,kind", eh.REGRESSION_NNFIELD)
def test_nnfield_unchanged_since_recorded(ctx, w, h, ns, nn, kind):
    g, t = np.load(eh.REGRESSION_FILE), eh.tag(w, h, ns, nn, kind)
    seeds, cost = nnfield_inputs(w, h, ns, kind)
    gl, gb, gd, _ = ctx.epic_nnfield(seeds, nn, cost)
    for name, a in (("labels_", gl), ("best_", gb), ("dist_", gd)):
        now, then = eh.stored(a), g[name + t]
        assert np.array_equal(now, then), "%s differs in %d of %d stored entries" % (name[:-1], int((now != then).sum()), then.size)


@pytest.mark.parametrize("w,h,n,method,filters", eh.REGRESSION_EPIC)
def test_epic_unchanged_since_recorded(ctx, w, h, n, method, filters):
    g, t = np.load(eh.REGRESSION_FILE), eh.tag(w, h, n, method, filters)
    ci, m, edges, p = epic_inputs(w, h, n, method, filters)
    gx, gy = Image(w, h), Image(w, h)
    st = ctx.epic(gx, gy, ci, m, edges, p)
    assert [st.matches_in, st.matches_after_saliency, st.matches_after_consistency] == g["counts_" + t].tolist()
    assert np.array_equal(eh.stored(edges, eh.FLOW_SAMPLE), g["edges_" + t])
    d = np.hypot(eh.stored(gx.array, eh.FLOW_SAMPLE) - g["fx_" + t], eh.stored(gy.array, eh.FLOW_SAMPLE) - g["fy_" + t])
    assert d.mean() <= 0.001 and d.max() <= 0.01, (d.mean(), d.max())
