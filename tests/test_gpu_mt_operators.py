"""The multi-frame path (Variational_MT) operator by operator against the C++ restatement oracle/sf_oracle_mt.cpp, whose
operator entries are the functions its pinned driver is made of (tests/test_oracle_pin_mt.py).

Every pixel is compared.  The interior and the band of 8 pixels along the borders are gated separately: the 99th
percentile of the relative error tightly and its maximum loosely.  The robust weights are 1 / sqrt(residual^2 + eps^2)
and friends, so a last-bit difference of a derivative is amplified where a residual vanishes: that is what the loose
maximum allows for.  Outputs are pre-filled with NaN, so every element has to be written, and the stride padding has to
hold zeros.  The gates sit a few times above the errors measured on a B200: the linear system 5.6e-6 (99th percentile)
and 3.3e-4 (maximum), the smoothness weights 4.6e-8 / 2.2e-7, the luminance weight 2.3e-7 / 4.6e-7, the occlusion costs
5.8e-7 / 2.4e-5 and the flow resampling 4.6e-7 (maximum)."""
import ctypes as C

import numpy as np
import pytest

import mt_helpers as mh
from slowflow_b200 import ColorImage, Context, Image
from oracle.pyoracle import SOR_REDBLACK

pytestmark = pytest.mark.gpu

FP, IP = C.POINTER(C.c_float), C.POINTER(C.c_int)
BAND = 8
VARIANTS = {"packed": {}, "scalar": {"SLOWFLOW_GPU_MT_TERMS_SCALAR": "1"}, "per_term": {"SLOWFLOW_GPU_MT_DATA_VARIANT": "1"}}


def gate(name, g, r, w, h, tight, loose, skip=None):
    """g: the GPU's Image, r: the reference's (height, width) array; skip: pixels not gated (a boolean mask).  The error
    of a pixel is taken relative to |r| + the plane's scale (the 99th percentile of |r|): the inverted blocks reach 1e6
    at the few pixels where neither a data term nor the smoothness holds the flow, and a scale set by those would hide
    errors everywhere else."""
    assert np.isfinite(g.full).all(), name + ": an element was not written"
    assert not g.full[:, w:].any(), name + ": stride padding"
    scale = float(np.percentile(np.abs(r), 99)) or 1.0
    err = np.abs(g.array.astype(np.float64) - r) / (np.abs(r) + scale)
    if skip is not None:
        err[skip] = 0.0
    border = np.ones((h, w), bool)
    border[BAND:-BAND, BAND:-BAND] = False
    out = []
    for region, sel in (("interior", ~border), ("border", border)):
        e = err[sel]
        if e.size == 0:
            continue
        p99, mx = float(np.percentile(e, 99)), float(e.max())
        out.append("%s %s p99 %.1e max %.1e" % (name, region, p99, mx))
        assert p99 <= tight, (name, region, p99, mx)
        assert mx <= loose, (name, region, p99, mx)
    print("; ".join(out))


def level(w, h, S, seed=20170721, leave=True):
    """frames of a window and a flow that leaves the image at a few pixels"""
    ims, wx, wy = mh.window(w, h, S, seed=seed)
    if leave:
        wx.array[3, 5] = -40.0
        wy.array[h - 2, w - 3] = 500.0
        wx.array[h // 2, w - 1] = 3.0 * w
    return ims, wx, wy


def normalised(oracle, ims, p):
    frames = [f.copy() for f in ims]
    q = mh.clone_params(p)
    oracle.lib.sfo_normalize(mh.frame_array(frames), len(frames), C.byref(q))
    return frames, q


def gpu_context(monkeypatch, variant):
    for k in ("SLOWFLOW_GPU_MT_TERMS_SCALAR", "SLOWFLOW_GPU_MT_DATA_VARIANT"):
        monkeypatch.delenv(k, raising=False)
    for k, v in VARIANTS[variant].items():
        monkeypatch.setenv(k, v)
    return Context(0)


# ------------------------------------------------------------------ the linear system of one linearisation
SYSTEM_CASES = {
    # name: (w, h, S, parameters, increment, channel weights)
    "modl1_17x13": (17, 13, 3, dict(), False, True),
    "geman_mcclure_66x31_S2_unnormalised": (66, 31, 2, dict(robust_color=4, robust_color_eps=0.5, dataterm=0, omega=[1]), True, False),
    "lorentzian_grad_gm_253x97": (253, 97, 3, dict(robust_color=2, robust_color_eps=0.5, robust_grad=4, robust_grad_eps=0.5), True, True),
    "trunc_modl1_253x97_S4_unnormalised": (253, 97, 4, dict(robust_color=3, robust_color_eps=0.001, robust_color_truncation=5.0,
                                                            dataterm=0, rho=[1, 1, 1], omega=[1, 2, 1]), False, True),
    "quadratic_2073x64_S6_unnormalised": (2073, 64, 6, dict(robust_color=0, robust_reg=2, robust_reg_eps=0.5, dataterm=0,
                                                            rho=[1, 1, 1, 1, 1], omega=[1, 2, 1, 1, 1]), True, True),
    "geman_mcclure_small_eps_61x45": (61, 45, 3, dict(robust_color=4, robust_color_eps=0.001), False, False),
    "separate_grad_lorentzian_96x64_S4": (96, 64, 4, dict(robust_grad=2, robust_grad_eps=0.5, rho=[1, 1, 1], omega=[0, 2, 1]), True, False),
    "one_direction_96x64_unnormalised": (96, 64, 3, dict(one_direction=1, dataterm=0, omega=[1, 2]), True, True),
    "geman_mcclure_1280x1024": (1280, 1024, 3, dict(robust_color=4, robust_color_eps=0.5), False, True),
}


def system_inputs(oracle, name):
    w, h, S, kw, increment, weighted = SYSTEM_CASES[name]
    ims, wx, wy = level(w, h, S)
    p = mh.params(S, hbit=0, **kw)
    frames, q = normalised(oracle, ims, p)
    rng = np.random.default_rng(len(name))
    occ = Image(w, h)
    occ.buf[:] = rng.choice(np.array([-1.0, 0.0, 1.0], np.float32), size=occ.buf.size)
    du = dv = chw = None
    if increment:
        du = Image.from_array(rng.uniform(-0.3, 0.3, size=(h, w)).astype(np.float32))
        dv = Image.from_array(rng.uniform(-0.3, 0.3, size=(h, w)).astype(np.float32))
    if weighted:
        chw = ColorImage.from_array(rng.uniform(0.5, 1.5, size=(3, h, w)).astype(np.float32))
    return dict(w=w, h=h, frames=frames, wx=wx, wy=wy, q=q, occ=occ, du=du, dv=dv, chw=chw)


_REFERENCE = {}


def system_reference(oracle, name):
    """sfo_mt_system, then the block inverse of the SOR's first sweep (sfo_sor_coupled inverts a11 / a12 / a22 in place)"""
    if name not in _REFERENCE:
        x = system_inputs(oracle, name)
        w, h = x["w"], x["h"]
        A = [Image(w, h) for _ in range(7)]
        rc = oracle.lib.sfo_mt_system(*[a.ptr() for a in A], mh.frame_array(x["frames"]), x["wx"].ptr(), x["wy"].ptr(),
                                      x["du"].ptr() if x["du"] else None, x["dv"].ptr() if x["dv"] else None, x["occ"].ptr(),
                                      x["chw"].ptr() if x["chw"] else None, C.byref(x["q"]))
        assert rc == 0
        inv = [a.copy() for a in A[:3]]
        z0, z1 = Image(w, h), Image(w, h)
        oracle.lib.sfo_sor_coupled(z0.ptr(), z1.ptr(), *[a.ptr() for a in inv], A[3].ptr(), A[4].ptr(), A[5].ptr(), A[6].ptr(), 1, 1.9,
                                   SOR_REDBLACK)
        _REFERENCE[name] = (x, [a.array.copy() for a in inv + A[3:]])
    return _REFERENCE[name]


def gpu_system(ctx, x):
    blocks, psi = ctx.mt_system(x["frames"], x["wx"], x["wy"], x["q"], x["occ"], x["du"], x["dv"], x["chw"])
    return blocks + psi


@pytest.mark.parametrize("variant", sorted(VARIANTS))
@pytest.mark.parametrize("name", sorted(SYSTEM_CASES))
def test_mt_system_matches_restatement(oracle, monkeypatch, name, variant):
    """One linearisation of compute_one_level through the production kernels: warps, derivative planes, luminance weight,
    smoothness, every data term with the occlusion factor and the channel weights, the Laplacian and the block inverse."""
    x, ref = system_reference(oracle, name)
    with gpu_context(monkeypatch, variant) as ctx:
        G = gpu_system(ctx, x)
    for k, label in enumerate(["a11'", "a12'", "a22'", "b1", "b2", "psi_h", "psi_v"]):
        gate("%s %s %s" % (name, variant, label), G[k], ref[k], x["w"], x["h"], 2e-5, 2e-3)


def test_mt_system_packed_kernel_runs(oracle, monkeypatch):
    """The packed all-terms kernel ran (it did not fall back to the scalar one): the two round differently."""
    x, _ = system_reference(oracle, "lorentzian_grad_gm_253x97")
    with gpu_context(monkeypatch, "packed") as ctx:
        a = gpu_system(ctx, x)
    with gpu_context(monkeypatch, "scalar") as ctx:
        b = gpu_system(ctx, x)
    assert any(not np.array_equal(p.full, s.full) for p, s in zip(a[:5], b[:5]))
    assert all(np.array_equal(p.full, s.full) for p, s in zip(a[5:], b[5:]))  # the smoothness pass is shared


# ------------------------------------------------------------------ occlusion data costs and their labelling
PENALTIES = {
    "quadratic": dict(robust_color=0),
    "modl1": dict(robust_color=1),
    "lorentzian": dict(robust_color=2, robust_color_eps=0.5),
    "trunc_modl1": dict(robust_color=3, robust_color_eps=0.001, robust_color_truncation=5.0),
    "geman_mcclure": dict(robust_color=4, robust_color_eps=0.5),
    "lorentzian_grad_gm": dict(robust_color=2, robust_color_eps=0.5, robust_grad=4, robust_grad_eps=0.5),
}


@pytest.mark.parametrize("S", [2, 3, 4])
@pytest.mark.parametrize("int_terms", [0, 1])
@pytest.mark.parametrize("penalty", sorted(PENALTIES))
def test_mt_occ_costs_match_restatement(ctx, oracle, penalty, int_terms, S):
    """k_occ_costs (the cost half of optimizeOcc) against the restatement, then the labelling of the GPU's costs: the
    restatement's min-cut and the device min-cut agree on them."""
    w, h = 131, 77
    ims, wx, wy = level(w, h, S, seed=S)
    p = mh.params(S, graphcut_int_terms=int_terms, rho=[1, 1, 1], omega=[1, 2, 1], **PENALTIES[penalty])
    frames, q = normalised(oracle, ims, p)
    g0, g1 = ctx.mt_occ_costs(frames, wx, wy, q)
    r0, r1 = Image(w, h), Image(w, h)
    assert oracle.lib.sfo_mt_occ_costs(r0.ptr(), r1.ptr(), mh.frame_array(frames), wx.ptr(), wy.ptr(), C.byref(q)) == 0
    for name, g, r in (("d0", g0, r0), ("d1", g1, r1)):
        assert np.isfinite(g.array).all(), name
        err = np.abs(g.array.astype(np.float64) - r.array)
        scale = float(np.abs(r.array).max())
        print("occ costs %s S=%d %s: p99 %.1e max %.1e" % (penalty, S, name, np.percentile(err, 99) / scale, err.max() / scale))
        assert np.percentile(err, 99) <= 2e-6 * scale and err.max() <= 1e-4 * scale, name
    d0, d1 = np.ascontiguousarray(g0.array).ravel(), np.ascontiguousarray(g1.array).ravel()
    L = oracle.lib
    L.sfo_mincut.argtypes = [C.c_int, C.c_int, FP, FP, C.c_float, C.c_int, IP]
    lab_cpu = np.full(w * h, -7, np.int32)
    assert L.sfo_mincut(w, h, d0.ctypes.data_as(FP), d1.ctypes.data_as(FP), C.c_float(q.occlusion_alpha), int_terms,
                        lab_cpu.ctypes.data_as(IP)) == 0
    lab_dev = np.full(w * h, -7, np.int32)
    stats = (C.c_int * 2)()
    rc = ctx.lib.sfgpu_grid_mincut_dev(ctx.h, w, h, d0.ctypes.data_as(FP), d1.ctypes.data_as(FP), C.c_float(q.occlusion_alpha),
                                       int_terms, lab_dev.ctypes.data_as(IP), stats)
    assert rc == 0, ctx.lib.sfgpu_last_error().decode()
    assert np.array_equal(lab_cpu, lab_dev)


# ------------------------------------------------------------------ smoothness with robust penalties
REG = {0: (0.001, 0.5), 1: (0.001, 0.5), 2: (0.5, 0.5), 3: (0.001, None), 4: (0.5, 0.5)}


def smoothness_arguments(uu, vv, mode):
    """the penalty's argument of every horizontal / vertical edge, as the restatement forms it (float32)"""
    u, v = uu.array.astype(np.float32), vv.array.astype(np.float32)
    h, w = u.shape
    half = np.float32(0.5)

    def d3(a, axis):  # 3-tap centred derivative with replicated borders (image.c convolve, order 1)
        pad = np.pad(a, [(1, 1) if ax == axis else (0, 0) for ax in range(2)], mode="edge")
        lo = pad[:-2] if axis == 0 else pad[:, :-2]
        hi = pad[2:] if axis == 0 else pad[:, 2:]
        return (np.float32(-0.5) * lo + np.float32(0.5) * hi).astype(np.float32)

    uy2, vy2, ux2, vx2 = d3(u, 0), d3(v, 0), d3(u, 1), d3(v, 1)
    th = np.zeros((h, w), np.float32)
    tv = np.zeros((h, w), np.float32)
    cu = half * (uy2[:, :-1] + uy2[:, 1:]) if mode else 0
    cv = half * (vy2[:, :-1] + vy2[:, 1:]) if mode else 0
    ux1, vx1 = u[:, 1:] - u[:, :-1], v[:, 1:] - v[:, :-1]
    th[:, :-1] = (ux1 * ux1 + cu * cu) + (vx1 * vx1 + cv * cv)
    cu = half * (ux2[:-1] + ux2[1:]) if mode else 0
    cv = half * (vx2[:-1] + vx2[1:]) if mode else 0
    uy1, vy1 = u[1:] - u[:-1], v[1:] - v[:-1]
    tv[:-1] = (uy1 * uy1 + cu * cu) + (vy1 * vy1 + cv * cv)
    return th, tv


@pytest.mark.parametrize("w,h", [(5, 5), (33, 9), (61, 45), (2073, 1166)])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("robust_reg", sorted(REG))
def test_mt_smoothness_robust_penalties(ctx, oracle, w, h, mode, robust_reg):
    """compute_smoothness of variational_aux_mt.cpp (modes 0 / 1) with every penalty.  The truncated modified L1 gets its
    threshold at the median edge, so that many edges lie near it; an edge whose argument is within 4 ulp of the threshold
    may round to either side and is the only one not gated."""
    rng = np.random.default_rng(w + 7 * mode + 31 * robust_reg)
    uu = Image.from_array(rng.uniform(-2, 2, size=(h, w)).astype(np.float32))
    vv = Image.from_array(rng.uniform(-2, 2, size=(h, w)).astype(np.float32))
    wgt = Image.from_array(rng.uniform(0.05, 0.5, size=(h, w)).astype(np.float32))
    eps, trunc = REG[robust_reg]
    th, tv = smoothness_arguments(uu, vv, mode)
    skip_h = skip_v = None
    if trunc is None:
        trunc = float(np.float32(np.sqrt(np.median(th[:, :-1]))))
        near = lambda t: np.abs(np.sqrt(t.astype(np.float64)) - trunc) <= 4 * np.spacing(np.float32(trunc))
        skip_h, skip_v = near(th), near(tv)
        assert (np.sqrt(th.astype(np.float64)) > trunc).any() and (np.sqrt(th.astype(np.float64)) < trunc).any()
    gh, gv, rh, rv = Image(w, h), Image(w, h), Image(w, h), Image(w, h)
    gh.buf[:] = np.nan
    gv.buf[:] = np.nan
    ctx.compute_smoothness(gh, gv, uu, vv, wgt, 4.0, robust_reg=robust_reg, eps=eps, trunc=trunc, mode=mode)
    assert oracle.lib.sfo_mt_smoothness(rh.ptr(), rv.ptr(), uu.ptr(), vv.ptr(), wgt.ptr(), 4.0, mode, robust_reg, eps, trunc) == 0
    tag = "smoothness %dx%d mode %d reg %d" % (w, h, mode, robust_reg)
    gate(tag + " psi_h", gh, rh.array, w, h, 5e-7, 2e-6, skip_h)
    gate(tag + " psi_v", gv, rv.array, w, h, 5e-7, 2e-6, skip_v)
    assert not gh.array[:, -1].any() and not gv.array[-1, :].any()


# ------------------------------------------------------------------ luminance weight of the de-normalised reference frame
@pytest.mark.parametrize("w,h", [(61, 45), (253, 97), (1280, 1024)])
@pytest.mark.parametrize("hbit,depth", [(0, 8), (1, 8), (1, 16)])
def test_mt_dpsis_weight_denormalised(ctx, oracle, w, h, hbit, depth):
    """compute_dpsis_weight of variational_aux_mt.cpp:673-719 on normalised frames with the avg / std normalize()
    published, the 8-bit (255) and 16-bit (65535) divisors, on 8-bit and 16-bit intensities."""
    ims, _, _ = mh.window(w, h, 3)
    if depth == 16:
        for f in ims:
            f.buf[:] = np.rint(f.buf * 257.0)
    frames, q = normalised(oracle, ims, mh.params(3, hbit=hbit))
    avg = (C.c_float * 3)(*q.img_norm_avg)
    std = (C.c_float * 3)(*q.img_norm_std)
    g, r = Image(w, h), Image(w, h)
    g.buf[:] = np.nan
    ctx.compute_dpsis_weight(g, frames[1], 5.0, list(q.img_norm_avg), list(q.img_norm_std), hbit)
    assert oracle.lib.sfo_mt_dpsis_weight(r.ptr(), frames[1].ptr(), 5.0, avg, std, hbit) == 0
    assert np.ptp(r.array) > 1e-4  # the weight varies over the frame (least on 8-bit data read as 16-bit)
    gate("dpsis %dx%d hbit %d %d-bit" % (w, h, hbit, depth), g, r.array, w, h, 1e-6, 2e-6)


# ------------------------------------------------------------------ flow resampling between pyramid levels
@pytest.mark.parametrize("w,h", [(250, 163), (2560, 1440)])
@pytest.mark.parametrize("p_scale", [0.9, 0.5])
def test_mt_flow_resampling_between_levels(ctx, oracle, w, h, p_scale):
    """niter_alter = 0: the solver leaves every level's flow alone, so the result is the pyramid's resampling chain alone --
    the flow taken down to the coarsest level and back up with the ratio of the level sizes as vector scale."""
    ims, wx, wy = mh.window(w, h, 3)
    p = mh.params(3, layers=3, p_scale=p_scale, niter_alter=0)
    g = mh.run_gpu(ctx, ims, wx, wy, p)
    r = mh.run_cpu(oracle.lib, "sfo_", ims, wx, wy, p, SOR_REDBLACK)
    assert g["stats"].levels == 3
    for a, b in (("wx", "wx"), ("wy", "wy")):
        ga, rb = g[a].array.astype(np.float64), r[b].array
        err = np.abs(ga - rb).max() / np.abs(rb).max()
        print("resampling %dx%d p_scale %.1f %s: max rel %.1e" % (w, h, p_scale, a, err))
        assert err <= 2e-6, (a, err)
    assert not np.array_equal(g["wx"].array, wx.array)  # the chain changed the flow
