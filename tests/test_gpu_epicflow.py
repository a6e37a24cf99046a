"""sfgpu_rgb_to_lab (k_rgb_to_lab) and sfgpu_epicflow_sequence (slowflow_b200/csrc/sf_epicflow.cu).

The Lab kernel is checked against a NumPy restatement of rgb_to_lab (image.c:694) with C's float / double promotions, against
OpenCV's own Lab conversion for the constants, and bit for bit against the reference's rgb_to_lab where it was built.  The
sequence entry must equal, pair by pair and bit for bit, rgb_to_lab -> epic -> variational on the same inputs."""
import ctypes as C

import numpy as np
import pytest

from slowflow_b200 import ColorImage, Image, synth
from slowflow_b200.api import EpicStats, FloatImage, epic_params_default, load_library
from slowflow_b200.image import color_image_t, image_t
from slowflow_b200.params import VariationalParams

pytestmark = pytest.mark.gpu

SENTINEL = np.float32(-12345.5)  # what the flow planes hold before a call (padding included)
STATS = ("matches_in", "matches_after_saliency", "matches_after_consistency", "sweeps_prefilter", "sweeps_interpolation")
f32, f64 = np.float32, np.float64


# ------------------------------------------------------------------------------------------------------- rgb_to_lab
def lab_restated(rgb):
    """rgb_to_lab of image.c:694 on a (3, ...) float32 array: float64 where C promotes, float32 where C stores."""
    with np.errstate(invalid="ignore", divide="ignore"):
        r, g, b = (rgb[c] / f32(255) for c in range(3))
        r, g, b = r.astype(f64), g.astype(f64), b.astype(f64)
        X = (0.412453 * r + 0.357580 * g + 0.180423 * b).astype(f32)
        Y = (0.212671 * r + 0.715160 * g + 0.072169 * b).astype(f32)
        Z = (0.019334 * r + 0.119193 * g + 0.950227 * b).astype(f32)
        X = (X.astype(f64) / 0.950456).astype(f32)
        Z = (Z.astype(f64) / 1.088754).astype(f32)
        T = f32(0.008856)
        Y3 = np.power(Y.astype(f64), 1. / 3).astype(f32)
        fX = np.where(X > T, np.power(X.astype(f64), 1. / 3), 7.787 * X.astype(f64) + 16 / 116.).astype(f32)
        fY = np.where(Y > T, Y3.astype(f64), 7.787 * Y.astype(f64) + 16 / 116.).astype(f32)
        fZ = np.where(Z > T, np.power(Z.astype(f64), 1. / 3), 7.787 * Z.astype(f64) + 16 / 116.).astype(f32)
        L = np.where(Y > T, (f32(116) * Y3).astype(f64) - 16.0, 903.3 * Y.astype(f64)).astype(f32)
        A, B = f32(500) * (fX - fY), f32(200) * (fY - fZ)
        q = ((L / f32(100)) * (L / f32(100))).astype(f64) - 0.6
        corr = np.exp(f64(-f32(1.5)) * (q * q)).astype(f32)
        return np.stack([L, A * corr, B * corr]), corr


def all_triples():
    """Every 8-bit RGB triple once, as a 4096 x 4096 image (3, 4096, 4096)."""
    i = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([(i >> 16) & 255, (i >> 8) & 255, i & 255]).astype(f32).reshape(3, 4096, 4096)


def special_values(w, h, seed=5):
    """A (3, h, stride) array -- padding columns included -- of zeros, 255, values around the threshold T (a grey value of
    about 2.26 puts Y at T; X and Z cross it near the same value) and random values in [0, 255]."""
    s = ((w + 3) // 4) * 4
    a = np.random.RandomState(seed).uniform(0, 255, (3, h, s)).astype(f32)
    flat = a.reshape(3, -1)
    k = flat.shape[1]
    q = max(1, k // 8)
    ramp = np.linspace(2.0, 2.6, 2 * q).astype(f32)

    def put(c, start, vals):
        n = max(0, min(vals.size, k - start))
        flat[c, start:start + n] = vals[:n]

    for c in range(3):
        put(c, 0, np.zeros(q, f32))
        put(c, q, np.full(q, 255, f32))
        put(c, 2 * q, ramp)  # grey ramp through T
        put(c, 4 * q + 2 * q * c, ramp)  # one channel at a time
    return a


def compare_lab(got, want):
    """-> (values that differ, values that differ by more than one float ulp)."""
    gi, wi = got.reshape(-1).view(np.int32).astype(np.int64), want.reshape(-1).view(np.int32).astype(np.int64)
    differ = gi != wi
    return int(differ.sum()), int((np.abs(gi - wi) > 1).sum())


def lab_on_device(ctx, full):
    """full: (3, h, stride) float32 incl. padding -> the device's Lab, (3, h, stride)."""
    _, h, s = full.shape
    src = ColorImage(s, h)  # width = stride: then the padding columns of the real width are ordinary columns
    src.buf[:] = full.reshape(-1)
    out = ctx.rgb_to_lab(src)
    return out.buf.reshape(3, h, s)


def test_lab_all_rgb_triples_against_restatement(ctx):
    rgb = all_triples()
    got = lab_on_device(ctx, rgb)
    want, _ = lab_restated(rgb)
    n, big = compare_lab(got, want)
    print("rgb_to_lab over 2^24 triples: %d of %d values differ from the restatement (all by 1 ulp: %s)" % (n, want.size, big == 0))
    assert big == 0 and n <= 1e-6 * want.size


@pytest.mark.parametrize("w,h", [(501, 333), (37, 29), (4, 3), (1, 1), (1023, 7)])
def test_lab_odd_widths_padding_and_special_values(ctx, w, h):
    full = special_values(w, h)
    src = ColorImage(w, h)
    src.buf[:] = full.reshape(-1)  # the padding columns hold values too: they are converted like every other column
    got = ctx.rgb_to_lab(src)
    assert (got.width, got.height, got.stride) == (w, h, src.stride)
    want, _ = lab_restated(full)
    n, big = compare_lab(got.buf, want)
    print("%dx%d: %d of %d values differ by 1 ulp" % (w, h, n, want.size))
    assert big == 0 and n <= max(1, 1e-6 * want.size)


def test_lab_constants_against_opencv(ctx):
    """L, a and b before the attenuation (c2 / corr, c3 / corr) agree with OpenCV's linear-RGB -> Lab conversion."""
    cv2 = pytest.importorskip("cv2")
    rgb = all_triples()[:, ::8, :]  # every 8th row of the triple image: 2^21 triples, every red and blue level
    got = lab_on_device(ctx, np.ascontiguousarray(rgb))
    corr = np.exp(-1.5 * ((got[0].astype(f64) / 100) ** 2 - 0.6) ** 2)
    # one pixel per row: OpenCV's vectorised path for wide rows approximates the cube root more coarsely (errors up to 3e-2)
    col = np.ascontiguousarray((rgb / 255.0).astype(f32).reshape(3, -1, 1).transpose(1, 2, 0))
    cv = cv2.cvtColor(col, cv2.COLOR_LRGB2Lab).transpose(2, 0, 1).reshape(rgb.shape)
    dL = np.abs(got[0] - cv[0]).max()
    da = np.abs(got[1] / corr - cv[1]).max()
    db = np.abs(got[2] / corr - cv[2]).max()
    print("against cv2 COLOR_LRGB2Lab: max |dL| %.2e, |da| %.2e, |db| %.2e" % (dL, da, db))
    assert dL <= 1e-3 and da <= 2e-2 and db <= 2e-2


def test_lab_against_reference_rgb_to_lab(ctx, reference):
    L = reference.lib
    if not hasattr(L, "rgb_to_lab"):
        pytest.skip("the reference build exports no rgb_to_lab")
    L.rgb_to_lab.argtypes = [C.POINTER(color_image_t)]
    L.rgb_to_lab.restype = C.POINTER(color_image_t)
    for w, h in [(640, 480), (501, 333), (37, 29)]:
        src = ColorImage(w, h)
        src.buf[:] = special_values(w, h, seed=w).reshape(-1)
        ref = L.rgb_to_lab(src.ptr()).contents
        P = src.stride * h
        want = np.concatenate([np.ctypeslib.as_array(p, (P,)).copy() for p in (ref.c1, ref.c2, ref.c3)])
        if hasattr(L, "color_image_delete"):
            L.color_image_delete.argtypes = [C.POINTER(color_image_t)]
            L.color_image_delete(C.byref(ref))
        got = ctx.rgb_to_lab(src)
        assert np.array_equal(got.buf.view(np.uint32), want.view(np.uint32)), "%dx%d: %d values differ" % (
            w, h, int((got.buf.view(np.uint32) != want.view(np.uint32)).sum()))


# ------------------------------------------------------------------------------------------------------- the sequence
def epic_params(method="LA", filters=True):
    p = epic_params_default()
    p.method = method.encode()
    if not filters:
        p.saliency_th, p.pref_nn = 0.0, 0
    return p


def sequence_inputs(w, h, counts, filters=True, seed=700):
    """-> (frames (n + 1 ColorImages in [0, 255]), matches, edges) of n = len(counts) consecutive pairs."""
    frames = [ColorImage.from_array(synth.frame(w, h, t, seed)) for t in range(len(counts) + 1)]
    ms, es = [], []
    for k, n in enumerate(counts):
        _, m, e = synth.epic_case(w, h, n, seed=seed + 31 * k, outliers=0.05 if filters else 0.0)
        ms.append(m)
        es.append(np.clip(e + 0.05 * np.random.RandomState(seed + k).rand(h, w), 0.0, 1.0).astype(f32))
    return frames, ms, es


def planes(w, h, n):
    out = []
    for _ in range(n):
        fx, fy = Image(w, h), Image(w, h)
        fx.buf[:], fy.buf[:] = SENTINEL, SENTINEL
        out.append((fx, fy))
    return out


def run_composition(ctx, frames, ms, es, ep, vp, pairs=None):
    """rgb_to_lab -> epic -> variational per pair, on copies of the edge maps."""
    w, h = frames[0].width, frames[0].height
    pairs = range(len(ms)) if pairs is None else pairs
    fl, eo, st = planes(w, h, len(pairs)), [], []
    for (fx, fy), k in zip(fl, pairs):
        e = es[k].copy()
        st.append(ctx.epic(fx, fy, ctx.rgb_to_lab(frames[k]), ms[k], e, ep))
        ctx.variational(fx, fy, frames[k], frames[k + 1], vp)
        eo.append(e)
    return fl, eo, st


def run_sequence(ctx, frames, ms, es, ep, vp, pinned=False):
    w, h = frames[0].width, frames[0].height
    fl, eo = planes(w, h, len(ms)), [e.copy() for e in es]
    bufs = [f.buf for f in frames] + [p.buf for f in fl for p in f] + eo
    if pinned:
        for b in bufs:
            assert ctx.lib.sfgpu_host_register(b.ctypes.data, b.nbytes) == 0
    try:
        st = ctx.epicflow_sequence(frames, ms, eo, [f[0] for f in fl], [f[1] for f in fl], ep, vp)
    finally:
        if pinned:
            for b in bufs:
                ctx.lib.sfgpu_host_unregister(b.ctypes.data)
    return fl, eo, st


def assert_same(a, b, first=0):
    (fa, ea, sa), (fb, eb, sb) = a, b
    for k in range(len(fb)):
        for name, x, y in (("flow x", fa[first + k][0].buf, fb[k][0].buf), ("flow y", fa[first + k][1].buf, fb[k][1].buf),
                           ("edges", ea[first + k], eb[k])):
            assert np.array_equal(x.view(np.uint32), y.view(np.uint32)), "pair %d: %s differs at %d entries" % (
                first + k, name, int((x.view(np.uint32) != y.view(np.uint32)).sum()))
        assert [getattr(sa[first + k], f) for f in STATS] == [getattr(sb[k], f) for f in STATS], "pair %d: stats differ" % (first + k)


def flow_params(delta=0.0, outer=5):
    vp = VariationalParams()
    load_library().variational_params_default(C.byref(vp))
    vp.delta, vp.niter_outer = delta, outer
    return vp


@pytest.mark.parametrize("w,h,counts,method,filters,vp,pinned", [
    (320, 200, [800], "LA", True, None, False),                    # one pair
    (320, 200, [800] * 5, "LA", True, None, False),
    (320, 200, [800] * 5, "NW", True, None, True),
    (320, 200, [800] * 5, "LA", False, None, False),                # filters off: no Lab planes are made
    (320, 200, [800] * 5, "NW", False, None, True),
    (501, 333, [2500] * 3, "LA", True, None, True),                 # odd width: stride != width
    (320, 200, [800, 90, 1500, 20, 300], "LA", True, None, False),  # mixed match counts (nns differs per pair)
    (320, 200, [800] * 4, "LA", True, (0.5, 3), True),              # delta != 0, 3 outer iterations
    (320, 200, [800] * 10, "LA", True, None, False),                # two chunks, pageable
    (320, 200, [800] * 10, "LA", True, None, True),                 # two chunks, page-locked
    (160, 120, [300] * 19, "NW", True, (0.0, 2), True),             # three chunks: every ring slot and buffer parity reused
])
def test_sequence_equals_composition(ctx, w, h, counts, method, filters, vp, pinned):
    frames, ms, es = sequence_inputs(w, h, counts, filters)
    ep = epic_params(method, filters)
    vp = None if vp is None else flow_params(*vp)
    want = run_composition(ctx, frames, ms, es, ep, vp)
    got = run_sequence(ctx, frames, ms, es, ep, vp, pinned)
    assert_same(got, want)
    moved = np.mean([np.abs(f[0].array).mean() for f in got[0]])
    print("%dx%d x %d pairs %s: consistency %s, mean |flow x| %.3f" % (w, h, len(counts), method,
                                                                      [s.matches_after_consistency for s in got[2]], moved))
    assert all(s.matches_after_consistency > 0 for s in got[2]) and moved > 0


def test_sequence_refuses_continue_from_previous(ctx):
    w, h = 64, 48
    frames, ms, es = sequence_inputs(w, h, [100, 100])
    ints = [np.ascontiguousarray(np.clip(f.array.transpose(1, 2, 0), 0, 255).astype(np.uint8)) for f in frames]
    fl = planes(w, h, 2)
    ctx.variational_sequence_int(ints, [f[0] for f in fl], [f[1] for f in fl])
    run_sequence(ctx, frames, ms, es, epic_params(), None)
    with pytest.raises(RuntimeError, match="continue_from_previous"):
        ctx.variational_sequence_int(ints[1:], [fl[0][0]], [fl[0][1]], continue_from_previous=True)


# ------------------------------------------------------------------------------------------------------- errors
def raw_sequence(ctx, n, frames, ms, es, fl, ep):
    """sfgpu_epicflow_sequence through ctypes; None entries become NULL pointers -> status."""
    IP, CP, FIP, FP = C.POINTER(image_t), C.POINTER(color_image_t), C.POINTER(FloatImage), C.POINTER(C.c_float)
    fm = [FloatImage(m.ctypes.data_as(FP), m.shape[1], m.shape[0]) if m is not None else None for m in ms]
    fe = [FloatImage(e.ctypes.data_as(FP), e.shape[1], e.shape[0]) for e in es]
    k = len(fl)
    return ctx.lib.sfgpu_epicflow_sequence(
        ctx.h, n, (CP * len(frames))(*[C.pointer(f.c) if f is not None else None for f in frames]),
        (FIP * k)(*[C.pointer(m) if m is not None else None for m in fm]), (FIP * k)(*[C.pointer(e) for e in fe]),
        C.byref(ep) if ep is not None else None, None, (IP * k)(*[C.pointer(f[0].c) for f in fl]),
        (IP * k)(*[C.pointer(f[1].c) for f in fl]), (EpicStats * k)())


def untouched(fl):
    return all((f[0].buf == SENTINEL).all() and (f[1].buf == SENTINEL).all() for f in fl)


def test_argument_errors_touch_nothing(ctx):
    w, h = 160, 120
    frames, ms, es = sequence_inputs(w, h, [300] * 3)
    ep = epic_params()
    err = lambda: ctx.lib.sfgpu_last_error().decode()

    def check(n=3, frames=frames, ms=ms, fl=None, ep=ep, words=()):
        fl = fl or planes(w, h, 3)
        eo = [e.copy() for e in es]
        assert raw_sequence(ctx, n, frames, ms, eo, fl, ep) == 2
        assert untouched(fl) and all(np.array_equal(a, b) for a, b in zip(eo, es)), err()
        for word in words:
            assert word in err(), err()

    check(n=0)
    check(ep=None)
    check(frames=frames[:1] + [None] + frames[2:], words=("pair 1", "null"))
    check(ms=ms[:2] + [None], words=("pair 2", "null"))
    check(ms=[ms[0], ms[1][:, :3].copy(), ms[2]], words=("pair 1", ">= 4 columns"))
    bad = planes(w, h, 3)
    bad[2] = (Image(w, h + 1), Image(w, h + 1))
    bad[2][0].buf[:], bad[2][1].buf[:] = SENTINEL, SENTINEL
    check(fl=bad, words=("pair 2",))
    other = ColorImage(w + 1, h)  # the last frame (only read by the refinement) has another geometry
    check(frames=frames[:3] + [other], words=("pair 2", "share width/height/stride"))
    odd = ColorImage(w, h)
    odd.c.c3 = odd.c.c2  # not planar-contiguous
    check(frames=[frames[0], odd] + frames[2:], words=("pair 0",))
    nw = epic_params()
    nw.method = b"XX"
    check(ep=nw, words=("method XX",))


def test_pair_without_matches_stops_at_its_chunk(ctx):
    """Pair 9 of 19 (chunk 1) has a flat first frame: its saliency is 0 everywhere and every match is removed.  Chunk 0 is
    complete, pairs 8..18 keep their planes, and chunk 2's edge maps are untouched."""
    w, h = 160, 120
    frames, ms, es = sequence_inputs(w, h, [300] * 19)
    frames[9] = ColorImage.from_array(np.zeros((3, h, w), f32))
    ep = epic_params()
    want = run_composition(ctx, frames, ms, es, ep, None, pairs=range(8))
    fl, eo = planes(w, h, 19), [e.copy() for e in es]
    with pytest.raises(RuntimeError, match=r"status 2\).*pair 9: no match survived the filters"):
        ctx.epicflow_sequence(frames, ms, eo, [f[0] for f in fl], [f[1] for f in fl], ep)
    assert untouched(fl[8:])
    for k in range(8):
        for name, x, y in (("flow x", fl[k][0].buf, want[0][k][0].buf), ("flow y", fl[k][1].buf, want[0][k][1].buf), ("edges", eo[k], want[1][k])):
            assert np.array_equal(x.view(np.uint32), y.view(np.uint32)), "pair %d: %s" % (k, name)
    assert all(np.array_equal(eo[k], es[k]) for k in range(16, 19))
