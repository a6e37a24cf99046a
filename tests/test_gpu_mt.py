"""Multi-frame (Variational_MT) parity on the GPU.

Checker: the reference's own unmodified driver (oracle/_ref: variational_mt.cpp + variational_aux_mt.cpp built
against header shims, SURVEY 8c) in its CPU red-black mode, and the C++ restatement oracle/sf_oracle_mt.cpp where
built.  Gate: mean endpoint difference <= 0.01 px, max <= 0.1 px, >= 8 px from the borders.  Non-convex penalties
are gated at eps = 0.5 (full iteration count) and over a short horizon at small eps (the reference iteration is
chaotic there, SURVEY 8d 'stability')."""
import numpy as np
import pytest

import mt_helpers as mh
from slowflow_b200 import ColorImage, Image, synth
from slowflow_b200.metrics import epe
from oracle.pyoracle import SOR_LEX, SOR_REDBLACK

pytestmark = pytest.mark.gpu
MEAN_TOL, MAX_TOL = 0.01, 0.1


def check(g, r, what, occ_frac_tol=0.002):
    mean, mx = epe(g["wx"].array, g["wy"].array, r["wx"].array, r["wy"].array, border=8)
    occ_diff = float((g["occ"].array != r["occ"].array).mean())
    print("%s: GPU vs CPU-RB mean %.3e max %.3e | occlusion labels differing %.4f%% | outer its gpu %d | avg change gpu %s cpu %s"
          % (what, mean, mx, 100 * occ_diff, g["stats"].outer_iterations, g["avg"], r["avg"]))
    assert mean <= MEAN_TOL and mx <= MAX_TOL, what
    assert occ_diff <= occ_frac_tol, what
    return mean, mx


def test_normalize_matches_reference(ctx, mt_checker):
    ims, wx, wy = mh.window(200, 120, 3)
    p = mh.params(3)
    r = mh.run_cpu(*mt_checker, ims, wx, wy, mh.params(3, niter_alter=1, niter_outer=1), SOR_REDBLACK)
    g_ims = [f.copy() for f in ims]
    ctx.normalize(g_ims, p)
    for k in range(3):
        assert abs(p.img_norm_avg[k] - r["params"].img_norm_avg[k]) <= 1e-4 * abs(r["params"].img_norm_avg[k])
        assert abs(p.img_norm_std[k] - r["params"].img_norm_std[k]) <= 1e-5
    for a, b in zip(g_ims, r["frames"]):
        assert np.abs(a.array - b.array).max() < 5e-4  # values ~ +-500 after normalisation


@pytest.mark.parametrize("name,kw", [
    ("modl1_default_occ", dict(niter_alter=2, niter_outer=4)),
    ("modl1_no_occ", dict(niter_alter=2, niter_outer=4, occlusion_reasoning=0)),
    ("geman_mcclure_eps0.5", dict(niter_alter=2, niter_outer=4, robust_color=4, robust_color_eps=0.5)),
    ("lorentzian_eps0.5_no_occ", dict(niter_alter=2, niter_outer=4, robust_color=2, robust_color_eps=0.5, occlusion_reasoning=0)),
    ("trunc_modl1_short", dict(niter_alter=1, niter_outer=2, robust_color=3, robust_color_eps=0.001, robust_color_truncation=5.0)),
    # quadratic data penalty: the reference iteration is unstable at the motion discontinuity (its own lex vs
    # red-black orderings differ by > 10 px after 3 outer iterations) -> gate the arithmetic over one iteration
    ("quadratic_reg_lorentzian_short", dict(niter_alter=1, niter_outer=1, robust_color=0, robust_reg=2, robust_reg_eps=0.5)),
    ("geman_mcclure_small_eps_short_horizon", dict(niter_alter=1, niter_outer=2, robust_color=4, robust_color_eps=0.001)),
    ("forward_only", dict(niter_alter=1, niter_outer=3, one_direction=1)),
    # slow_flow_dataterm = 0: the reference-term branch carries copy-paste slips (SURVEY Q5, reproduced literally)
    # that make the reference itself blow up after 2 outer iterations -> one iteration with them, two without
    ("unnormalised_dataterm_short", dict(niter_alter=1, niter_outer=1, dataterm=0)),
    ("unnormalised_dataterm_succ_only", dict(niter_alter=1, niter_outer=2, dataterm=0, omega=[0, 0])),
    ("smoothing0_inner2", dict(niter_alter=1, niter_outer=2, niter_inner=2, smoothing=0)),
    ("separate_grad_penalty", dict(niter_alter=1, niter_outer=2, robust_grad=2, robust_grad_eps=0.5)),
    # 16bit = 1 is what the shipped cfgs/slow_flow.cfg and sf_mt_params_default select: the smoothness weight divides the
    # de-normalised luminance by 65535 (variational_aux_mt.cpp:673-719).  Once on 16-bit intensities (0..65535), once on
    # 8-bit intensities (the flat-weight case a user gets who leaves the flag at its default)
    ("hbit16_modl1_occ", dict(niter_alter=2, niter_outer=4, hbit=1)),
    ("hbit16_geman_mcclure_eps0.5", dict(niter_alter=2, niter_outer=3, hbit=1, robust_color=4, robust_color_eps=0.5)),
    ("hbit_flag_on_8bit_data", dict(niter_alter=2, niter_outer=3, hbit=1)),
])
def test_mt_parity_small(ctx, mt_checker, name, kw):
    ims, wx, wy = mh.window(256, 160, 3)
    if name.startswith("hbit16"):
        for f in ims:
            f.buf[:] = np.rint(f.buf * 257.0)  # 0..255 -> 0..65535, integer valued like a 16-bit image
    p = mh.params(3, **kw)
    r = mh.run_cpu(*mt_checker, ims, wx, wy, p, SOR_REDBLACK)
    g = mh.run_gpu(ctx, ims, wx, wy, p)
    check(g, r, name)


def test_mt_parity_S2_and_S4(ctx, mt_checker):
    for S in (2, 4):
        ims, wx, wy = mh.window(192, 128, S)
        p = mh.params(S, niter_alter=2, niter_outer=3, rho=[1, 1, 1], omega=[0, 2, 1])
        r = mh.run_cpu(*mt_checker, ims, wx, wy, p, SOR_REDBLACK)
        g = mh.run_gpu(ctx, ims, wx, wy, p)
        check(g, r, "S=%d" % S)


def test_mt_parity_S6_more_frames_than_one_warp_launch_takes(ctx, mt_checker):
    """S = 6: 10 warped frames, i.e. two launches of the batched warp + derivative kernel (8 frames per launch,
    sf_wderivs.cu)."""
    S = 6
    ims, wx, wy = mh.window(160, 96, S)
    p = mh.params(S, niter_alter=1, niter_outer=2, rho=[1, 1, 1, 1, 1], omega=[0, 2, 1, 1, 1])
    r = mh.run_cpu(*mt_checker, ims, wx, wy, p, SOR_REDBLACK)
    g = mh.run_gpu(ctx, ims, wx, wy, p)
    check(g, r, "S=%d" % S)


def test_mt_pyramid_three_layers_zero_init(ctx, mt_checker):
    """Config 4 in small: layers = 3, p_scale = 0.9, zero initial flow, odd level widths (stride != width)."""
    ims, wx, wy = mh.window(250, 163, 3, zero_flow=True)
    p = mh.params(3, layers=3, niter_alter=1, niter_outer=3)
    r = mh.run_cpu(*mt_checker, ims, wx, wy, p, SOR_REDBLACK)
    g = mh.run_gpu(ctx, ims, wx, wy, p)
    assert g["stats"].levels == 3
    check(g, r, "pyramid 3 layers")


def test_mt_config3_1280x1024(ctx, mt_checker):
    """BASELINE config 3 geometry (1280x1024, S=3, 5 frames) with Geman-McClure eps=0.5, occlusion reasoning on,
    bounded to 2 alternations x 3 outer iterations so the CPU reference finishes in about a minute."""
    ims, wx, wy = mh.window(1280, 1024, 3)
    p = mh.params(3, niter_alter=2, niter_outer=3, robust_color=4, robust_color_eps=0.5)
    r = mh.run_cpu(*mt_checker, ims, wx, wy, p, SOR_REDBLACK)
    g = mh.run_gpu(ctx, ims, wx, wy, p)
    check(g, r, "config 3 (bounded)")
    lex = mh.run_cpu(*mt_checker, ims, wx, wy, p, SOR_LEX)
    print("reported: GPU vs CPU-lex mean %.3e max %.3e" % epe(g["wx"].array, g["wy"].array, lex["wx"].array, lex["wy"].array))


def test_mt_config3_full_iteration_count(ctx, mt_checker, oracle):
    """BASELINE config 3 with its FULL iteration count: 1280x1024, S=3, Geman-McClure eps 0.5, occlusion reasoning,
    2 alternations x 10 outer iterations x 30 SOR sweeps against the reference's own unmodified driver (CPU red-black).
    The executed outer-iteration counts must agree too (the early exits of variational_mt.cpp:407,436)."""
    ims, wx, wy = mh.window(1280, 1024, 3)
    p = mh.params(3, niter_alter=2, niter_outer=10, robust_color=4, robust_color_eps=0.5)
    r = mh.run_cpu(*mt_checker, ims, wx, wy, p, SOR_REDBLACK)
    g = mh.run_gpu(ctx, ims, wx, wy, p)
    check(g, r, "config 3 (2 x 10 outer iterations)")
    assert abs(g["avg"][0] - r["avg"][0]) < 1e-4 and abs(g["avg"][1] - r["avg"][1]) < 1e-4
    # the reference driver does not count its iterations; the restatement (bit-identical to it, test_oracle_pin_mt.py) does
    o = mh.run_cpu(oracle.lib, "sfo_", ims, wx, wy, p, SOR_REDBLACK)
    print("outer iterations executed: gpu %d, cpu %d" % (g["stats"].outer_iterations, o["stats"][0]))
    assert g["stats"].outer_iterations == o["stats"][0]


def test_mt_early_exit_iteration_counts(ctx, mt_checker):
    """Convergent setting: the early exits (variational_mt.cpp:407,436) must fire on the GPU as on the CPU."""
    ims, wx, wy = mh.window(160, 120, 2)
    p = mh.params(2, niter_alter=3, niter_outer=10, thres_outer=5e-3, occlusion_reasoning=0)
    r = mh.run_cpu(*mt_checker, ims, wx, wy, p, SOR_REDBLACK)
    g = mh.run_gpu(ctx, ims, wx, wy, p)
    check(g, r, "early exit")
    assert g["stats"].outer_iterations < 30
    assert abs(g["avg"][0] - r["avg"][0]) < 1e-4 and abs(g["avg"][1] - r["avg"][1]) < 1e-4


def test_mt_class_shape(ctx):
    """Variational_MT mirror (variational_mt.h:23-71): setChannelWeights / getOcclusions / one_direction."""
    from slowflow_b200 import ColorImage, Variational_MT
    ims, wx, wy = mh.window(128, 96, 2)
    p = mh.params(2, niter_alter=1, niter_outer=2)
    solver = Variational_MT(ctx)
    w = ColorImage(128, 96)
    w.buf[:] = 1.0
    solver.setChannelWeights(w)
    a, b = wx.copy(), wy.copy()
    r1 = solver.variational(a, b, ims, p)
    plain = Variational_MT(ctx)
    c, d = wx.copy(), wy.copy()
    r2 = plain.variational(c, d, ims, p)
    assert np.array_equal(a.array, c.array) and r1 == r2  # all-ones weights == no weights
    assert solver.getOcclusions() is not None and set(np.unique(solver.getOcclusions().array)) <= {-1.0, 0.0, 1.0}


def test_mt_gpu_vs_restatement(ctx, oracle):
    """Same gate against the C++ restatement (the checker that always travels as source)."""
    ims, wx, wy = mh.window(200, 144, 3)
    p = mh.params(3, niter_alter=2, niter_outer=3, robust_color=2, robust_color_eps=0.5)
    r = mh.run_cpu(oracle.lib, "sfo_", ims, wx, wy, p, SOR_REDBLACK)
    g = mh.run_gpu(ctx, ims, wx, wy, p)
    check(g, r, "vs restatement")


# ------------------------------------------------------------------ input side of a window (SURVEY 8f rank 3)
@pytest.mark.parametrize("w,h,scale", [(131, 97, 0.5), (200, 150, 0.75), (97, 61, 0.9), (64, 48, 0.3), (80, 60, 1.5)])
def test_prescale_matches_oracle(ctx, oracle, w, h, scale):
    """GaussianBlur + resize by factor (slow_flow.cpp:538-542) against the restatement pinned to cv2."""
    import ctypes as C
    from slowflow_b200 import ColorImage
    from slowflow_b200.image import color_image_t
    r = np.random.RandomState(w)
    src = ColorImage.from_array((r.rand(3, h, w) * 255).astype(np.float32))
    g = ctx.prescale(src, scale)
    L = oracle.lib
    CP = C.POINTER(color_image_t)
    L.sfo_prescale.argtypes = [CP, CP, C.c_float]
    ref = ColorImage(g.width, g.height)
    assert L.sfo_prescale(ref.ptr(), src.ptr(), scale) == 0
    assert (g.width, g.height) == (int(np.rint(w * np.float64(np.float32(scale)))), int(np.rint(h * np.float64(np.float32(scale)))))
    assert np.abs(g.array - ref.array).max() <= 2e-4  # values up to 255: fp32 FMA contraction only


@pytest.mark.parametrize("red_x,red_y,weight", [(0, 0, 1.0), (1, 0, 2.0), (0, 1, 0.5), (1, 1, 3.7), (1, 1, -1.0)])
def test_raw_weighting_matches_oracle(ctx, oracle, red_x, red_y, weight):
    """rawWeighting (utils/utils.cpp:1336-1374) is pure index logic: bit-exact, padding untouched."""
    import ctypes as C
    from slowflow_b200 import ColorImage
    from slowflow_b200.image import color_image_t
    w, h = 37, 22
    a, b = ColorImage(w, h), ColorImage(w, h)
    a.buf[:] = -5.0
    b.buf[:] = -5.0
    ctx.raw_weighting(a, red_x, red_y, weight)
    L = oracle.lib
    L.sfo_raw_weighting.argtypes = [C.POINTER(color_image_t), C.c_int, C.c_int, C.c_float]
    assert L.sfo_raw_weighting(b.ptr(), red_x, red_y, weight) == 0
    assert np.array_equal(a.buf, b.buf)
    assert np.allclose(a.array.sum(axis=0), 3.0)  # the three weights of a pixel always add up to 3


def test_normalize_streaming_path_equals_resident(ctx, monkeypatch):
    """Long sequences are normalised through one frame-sized device buffer (two passes); same result as resident."""
    ims, _, _ = mh.window(120, 80, 3)
    a, b = [f.copy() for f in ims], [f.copy() for f in ims]
    pa, pb = mh.params(3), mh.params(3)
    ctx.normalize(a, pa)
    monkeypatch.setenv("SLOWFLOW_GPU_NORMALIZE_RESIDENT_BYTES", "0")
    ctx.normalize(b, pb)
    for x, y in zip(a, b):
        assert np.array_equal(x.array, y.array)
    assert list(pa.img_norm_avg) == list(pb.img_norm_avg) and list(pa.img_norm_std) == list(pb.img_norm_std)


def test_mt_config4_2560x1440_three_layers_bounded(ctx, mt_checker):
    """BASELINE config 4 geometry: 2560x1440, zero initial flow, 3 pyramid layers (2560x1440 -> 2304x1296 -> 2073x1166,
    stride 2076), bounded to one outer iteration per level so that the CPU reference finishes in about a minute."""
    ims, wx, wy = mh.window(2560, 1440, 3, zero_flow=True)
    p = mh.params(3, layers=3, niter_alter=1, niter_outer=1, robust_color=4, robust_color_eps=0.5)
    r = mh.run_cpu(*mt_checker, ims, wx, wy, p, SOR_REDBLACK)
    g = mh.run_gpu(ctx, ims, wx, wy, p)
    assert g["stats"].levels == 3
    check(g, r, "config 4 (bounded)")


def test_mt_data_pass_variants_agree(monkeypatch):
    """The default multi-frame data pass (per-frame derivative planes + one pointwise all-terms kernel) against the
    one-fused-kernel-per-term variant (SLOWFLOW_GPU_MT_DATA_VARIANT=1): the two differ only in where the linear
    combination of the two frames of a term is taken (before or after the derivative filters), i.e. in rounding."""
    from slowflow_b200 import Context
    ims, wx, wy = mh.window(300, 190, 3)
    p = mh.params(3, niter_alter=2, niter_outer=3, robust_color=4, robust_color_eps=0.5)
    with Context(0) as c0:
        a = mh.run_gpu(c0, ims, wx, wy, p)
    monkeypatch.setenv("SLOWFLOW_GPU_MT_DATA_VARIANT", "1")
    with Context(0) as c1:
        b = mh.run_gpu(c1, ims, wx, wy, p)
    mean, mx = epe(a["wx"].array, a["wy"].array, b["wx"].array, b["wy"].array, border=0)
    print("fused vs per-term data pass: mean %.3e max %.3e" % (mean, mx))
    assert mean <= 1e-4 and mx <= 1e-2
    assert float((a["occ"].array != b["occ"].array).mean()) <= 0.002


@pytest.mark.parametrize("kw", [
    dict(robust_color=4, robust_color_eps=0.5),
    dict(robust_color=1),
    dict(robust_color=2, robust_color_eps=0.5, robust_grad=4, robust_grad_eps=0.5),
    dict(robust_color=3, robust_color_eps=0.001, robust_color_truncation=5.0),
    # quadratic data penalty: unstable reference iteration (see test_mt_parity_small) -> the arithmetic over one iteration
    dict(robust_color=0, robust_reg=2, robust_reg_eps=0.5, niter_alter=1, niter_outer=1),
    # slow_flow_dataterm = 0 with reference terms: the reference's own slips blow the iteration up after 2 outer iterations
    dict(dataterm=0, niter_alter=1, niter_outer=1),
    dict(dataterm=0, omega=[0, 0], niter_inner=2),
    dict(one_direction=1, niter_inner=2),
])
def test_mt_terms_packed_vs_scalar(monkeypatch, kw):
    """The all-terms pass with two columns per thread on the packed pipe (k_mt_terms2, the default) against the
    one-column-per-thread kernel with the scalar term functions (SLOWFLOW_GPU_MT_TERMS_SCALAR=1), on an ODD width
    (the last pair of a row is pixel + padding), with channel weights, over every penalty and both dataterm branches."""
    from slowflow_b200 import Context
    w, h = 253, 97
    ims, wx, wy = mh.window(w, h, 3)
    rng = np.random.default_rng(5)
    chw = ColorImage.from_array(rng.uniform(0.5, 1.5, size=(3, h, w)).astype(np.float32))
    p = mh.params(3, **{**dict(niter_alter=2, niter_outer=2), **kw})
    with Context(0) as c0:
        a = mh.run_gpu(c0, ims, wx, wy, p, chw)
    monkeypatch.setenv("SLOWFLOW_GPU_MT_TERMS_SCALAR", "1")
    with Context(0) as c1:
        b = mh.run_gpu(c1, ims, wx, wy, p, chw)
    assert np.isfinite(a["wx"].array).all() and np.isfinite(a["wy"].array).all()
    mean, mx = epe(a["wx"].array, a["wy"].array, b["wx"].array, b["wy"].array, border=0)
    moved = float(np.abs(a["wx"].array - wx.array).mean())
    print("packed vs scalar terms %s: mean %.3e max %.3e (moved %.3f)" % (kw, mean, mx, moved))
    assert moved > 1e-3
    assert mean <= 1e-4 and mx <= 1e-2


def test_mt_channel_weights_parity(ctx, mt_checker):
    """channel_w (the rawWeighting planes, variational_mt.cpp:343-361) through the default all-terms pass against the
    reference driver, on an odd width."""
    w, h = 253, 131
    ims, wx, wy = mh.window(w, h, 3)
    rng = np.random.default_rng(11)
    chw = ColorImage.from_array(rng.uniform(0.5, 1.5, size=(3, h, w)).astype(np.float32))
    p = mh.params(3, niter_alter=2, niter_outer=3, robust_color=4, robust_color_eps=0.5)
    r = mh.run_cpu(*mt_checker, ims, wx, wy, p, SOR_REDBLACK, chw)
    g = mh.run_gpu(ctx, ims, wx, wy, p, chw)
    check(g, r, "channel weights")


def test_mt_channel_weights_on_a_coarser_level(ctx, mt_checker):
    """layers = 2 with channel weights: the coarser level reads the level-0 weight planes with its own stride, like the
    reference does (it never rescales the weights, SURVEY Q14)."""
    w, h = 253, 131
    ims, wx, wy = mh.window(w, h, 3)
    rng = np.random.default_rng(12)
    chw = ColorImage.from_array(rng.uniform(0.5, 1.5, size=(3, h, w)).astype(np.float32))
    p = mh.params(3, layers=2, niter_alter=2, niter_outer=3, robust_color=4, robust_color_eps=0.5)
    r = mh.run_cpu(*mt_checker, ims, wx, wy, p, SOR_REDBLACK, chw)
    g = mh.run_gpu(ctx, ims, wx, wy, p, chw)
    assert g["stats"].levels == 2
    check(g, r, "channel weights, 2 layers")


@pytest.mark.parametrize("w,h", [(17, 13), (33, 9), (66, 31), (127, 40)])
def test_mt_tiny_and_ragged_windows(monkeypatch, w, h):
    """Ragged widths around the 64-column tile of the packed all-terms pass and the 56-column strips of the marching
    kernels, images smaller than one tile: finite results, packed and scalar terms agree."""
    from slowflow_b200 import Context
    ims, wx, wy = mh.window(w, h, 3)
    p = mh.params(3, niter_alter=2, niter_outer=2, robust_color=4, robust_color_eps=0.5)
    with Context(0) as c0:
        a = mh.run_gpu(c0, ims, wx, wy, p)
    monkeypatch.setenv("SLOWFLOW_GPU_MT_TERMS_SCALAR", "1")
    with Context(0) as c1:
        b = mh.run_gpu(c1, ims, wx, wy, p)
    assert np.isfinite(a["wx"].array).all() and np.isfinite(a["wy"].array).all()
    mean, mx = epe(a["wx"].array, a["wy"].array, b["wx"].array, b["wy"].array, border=0)
    print("tiny window %dx%d: packed vs scalar mean %.3e max %.3e" % (w, h, mean, mx))
    assert mean <= 1e-4 and mx <= 1e-2


def test_mt_frame_cache_same_results():
    """sfgpu_mt_frame_cache: consecutive windows over one sequence (sharing frames, forward and reversed order like the jet
    loop of slow_flow.cpp:875-1030) give bit-identical flows with and without the device-side frame cache; a change of
    geometry and re-enabling after the caller changed a frame are handled."""
    from slowflow_b200 import Context
    S, w, h = 3, 190, 110
    frames, _, _ = synth.window_case(w, h, 5, 20170721, 0.25, True)  # 9 frames: windows of 5 at offsets 0, 2, 4
    seq = [ColorImage.from_array(f) for f in frames]
    p = mh.params(S, niter_alter=2, niter_outer=2, robust_color=4, robust_color_eps=0.5)

    def solve_all(ctx):
        out = []
        q = mh.clone_params(p)
        ims = [f.copy() for f in seq]
        ctx.normalize(ims, q)
        for off in (0, 2, 4):
            for win in (ims[off:off + 5], ims[off:off + 5][::-1]):
                wx, wy, occ = Image(w, h), Image(w, h), Image(w, h)
                ctx.variational_mt(wx, wy, win, q, None, occ)
                out.append((wx.array.copy(), wy.array.copy(), occ.array.copy()))
        return out, ims, q

    with Context(0) as c0:
        plain, _, _ = solve_all(c0)
    with Context(0) as c1:
        c1.mt_frame_cache(7)
        cached, ims, q = solve_all(c1)
        for a, b in zip(plain, cached):
            for x, y in zip(a, b):
                assert np.array_equal(x, y)
        # another geometry through the same cache, then the first one again
        ims2, wx2, wy2 = mh.window(97, 61, S)
        g2 = mh.run_gpu(c1, ims2, wx2, wy2, p)
        assert np.isfinite(g2["wx"].array).all()
        wx, wy = Image(w, h), Image(w, h)
        c1.variational_mt(wx, wy, ims[0:5], q, None, None)
        assert np.array_equal(wx.array, plain[0][0])
        # the caller changes a frame: re-enabling empties the cache, the new contents are used
        ims[2].buf[:] = ims[2].buf * 0.5
        c1.mt_frame_cache(7)
        wx, wy = Image(w, h), Image(w, h)
        c1.variational_mt(wx, wy, ims[0:5], q, None, None)
    with Context(0) as c2:
        rx, ry = Image(w, h), Image(w, h)
        c2.variational_mt(rx, ry, ims[0:5], q, None, None)
    assert np.array_equal(wx.array, rx.array) and np.array_equal(wy.array, ry.array)
    assert not np.array_equal(rx.array, plain[0][0])
