"""sfgpu_slow_flow_jets against the composition it replaces, built from the existing entries: integer frame -> float32 ->
ctx.prescale (scale != 1) -> ctx.normalize over all frames -> Variational_MT per window -> x steps in float32.  Every
output plane is compared bit for bit, stride padding included, together with the published img_norm_* and the summed
outer-iteration count of sfgpu_get_mt_stats."""
import contextlib
import ctypes as C
import mmap

import numpy as np
import pytest

from slowflow_b200 import ColorImage, Image, Variational_MT, mt_params_default, synth
from slowflow_b200.api import FrameInt
from slowflow_b200.image import ceil4, image_t
from slowflow_b200.params import MTParams

pytestmark = pytest.mark.gpu

SENTINEL = np.float32(-12345.5)
IP = C.POINTER(image_t)


def params(S, **kw):
    p = mt_params_default()
    p.S = S
    p.hbit = 0
    p.niter_alter, p.niter_outer, p.niter_solver = 2, 4, 20
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def clone(p):
    return MTParams.from_buffer_copy(bytes(p))


def own_pages(shape, dtype):
    """A zeroed array on pages no other array uses (so that it can be page-locked on its own)."""
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    raw = np.zeros(nbytes + 2 * mmap.PAGESIZE, np.uint8)
    off = (-raw.ctypes.data) % mmap.PAGESIZE
    return raw[off:off + nbytes].view(dtype).reshape(shape)


def int_frames(w, h, n, dtype=np.uint8, channels=3, top=255, pad=0, seed=20170721, t0=0.0):
    """n frames of the moving synthetic texture as (H, W, channels) cv::Mat-like views with `pad` spare samples per row."""
    out = []
    for t in range(n):
        f = np.rint(synth.frame(w, h, t0 + 0.7 * t, seed) * (top / 255.0)).clip(0, top).astype(dtype)  # (3, H, W)
        canvas = own_pages((h, w + pad, channels), dtype)
        canvas[:, :w, :] = np.moveaxis(f, 0, 2)[:, :, :channels]
        out.append(canvas[:, :w, :] if channels == 3 else canvas[:, :w, 0])
    return out


def composition(ctx, frames, p, n_jets, first_jet=0, scale=1.0, back_one=False, channel_w=None):
    steps = p.S - 1
    ims = []
    for f in frames:
        a = f.astype(np.float32)
        a = np.stack([a] * 3) if a.ndim == 2 else np.moveaxis(a, 2, 0)
        im = ColorImage.from_array(a)
        ims.append(ctx.prescale(im, scale) if scale != 1.0 else im)
    q = clone(p)
    ctx.normalize(ims, q)
    w, h = ims[0].width, ims[0].height
    fwd, back, occ, outer = [], [], [], 0
    for j in range(first_jet, first_jet + n_jets):
        b = j * steps
        m = Variational_MT(ctx)
        m.setChannelWeights(channel_w)
        wx, wy = Image(w, h), Image(w, h)
        m.variational(wx, wy, ims[b:b + 2 * steps + 1], q)
        outer += ctx.mt_stats().outer_iterations
        fwd.append((wx.buf * np.float32(steps), wy.buf * np.float32(steps)))
        occ.append(m.getOcclusions().buf.copy())
        m = Variational_MT(ctx)
        m.one_direction = back_one
        wx, wy = Image(w, h), Image(w, h)
        m.variational(wx, wy, [ims[b + 3 * steps - i] for i in range(2 * steps + 1)], q)
        outer += ctx.mt_stats().outer_iterations
        back.append((wx.buf * np.float32(steps), wy.buf * np.float32(steps)))
    return dict(params=q, fwd=fwd, back=back, occ=occ, outer=outer)


def jets(ctx, frames, p, n_jets, **kw):
    q = clone(p)
    fwd, back, occ = ctx.slow_flow_jets(frames, q, n_jets, occlusions=True, **kw)
    return dict(params=q, fwd=[(x.buf, y.buf) for x, y in fwd], back=[(x.buf, y.buf) for x, y in back], occ=[o.buf for o in occ],
                outer=ctx.mt_stats().outer_iterations)


def same(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def assert_equal(got, want, outer=True):
    assert list(got["params"].img_norm_avg) == list(want["params"].img_norm_avg)
    assert list(got["params"].img_norm_std) == list(want["params"].img_norm_std)
    for kind in ("fwd", "back"):
        assert len(got[kind]) == len(want[kind])
        for k, (g, w) in enumerate(zip(got[kind], want[kind])):
            assert same(g[0], w[0]) and same(g[1], w[1]), "%s jet %d differs" % (kind, k)
    for k, (g, w) in enumerate(zip(got["occ"], want["occ"])):
        assert same(g, w), "occlusions of jet %d differ" % k
    if outer:
        assert got["outer"] == want["outer"]


CASES = {
    "u8_rgb_S2_occlusions": dict(shape=(96, 64), S=2, n_jets=3, kw=dict(occlusion_reasoning=1)),
    "u16_rgb_padded_step_S3_hbit": dict(shape=(96, 64), S=3, n_jets=2, dtype=np.uint16, top=4095, pad=3, kw=dict(hbit=1)),
    "u8_grey_odd_width": dict(shape=(77, 61), S=2, n_jets=2, channels=1),
    "scale_half": dict(shape=(130, 100), S=2, n_jets=2, scale=0.5),
    "two_layers": dict(shape=(96, 64), S=2, n_jets=2, kw=dict(layers=2, p_scale=0.8)),
    "backward_one_direction": dict(shape=(96, 64), S=2, n_jets=2, back_one=True),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_jets_equal_composition(ctx, name):
    c = CASES[name]
    w, h = c["shape"]
    steps = c["S"] - 1
    frames = int_frames(w, h, 1 + (c["n_jets"] + 2) * steps, c.get("dtype", np.uint8), c.get("channels", 3), c.get("top", 255),
                        c.get("pad", 0))
    p = params(c["S"], **c.get("kw", {}))
    scale, back_one = c.get("scale", 1.0), c.get("back_one", False)
    want = composition(ctx, frames, p, c["n_jets"], scale=scale, back_one=back_one)
    got = jets(ctx, frames, p, c["n_jets"], scale=scale, backward_one_direction=back_one)
    if scale != 1.0:
        assert got["fwd"][0][0].size == ceil4(round(w * scale)) * round(h * scale)
    assert all(np.isfinite(x).all() for f in got["fwd"] for x in f)
    assert np.abs(got["fwd"][0][0]).max() > 0.05  # the windows moved the flow
    assert_equal(got, want)


def test_jets_channel_weights(ctx):
    w, h = 96, 64
    frames = int_frames(w, h, 4 + 1 + 1, seed=11)  # S = 2: jets 0 and 1 need 5 frames
    cw = ColorImage(w, h)
    cw.buf[:] = 1.0
    ctx.raw_weighting(cw, 1, 0, 2.0)
    p = params(2)
    assert_equal(jets(ctx, frames, p, 2, channel_w=cw), composition(ctx, frames, p, 2, channel_w=cw))


def test_jets_statistics_cover_every_frame(ctx):
    """Frames beyond the last jet's window change the normalisation and therefore the results."""
    w, h = 96, 64
    frames = int_frames(w, h, 12, seed=5)
    frames[10] = (frames[10] // 3).astype(np.uint8)
    frames[11] = np.full_like(frames[11], 250)
    p = params(2)
    got = jets(ctx, frames, p, 2)
    assert_equal(got, composition(ctx, frames, p, 2))
    short = jets(ctx, frames[:5], p, 2)
    assert list(short["params"].img_norm_avg) != list(got["params"].img_norm_avg)


def test_jets_first_jet_shards(ctx):
    w, h = 96, 64
    frames = int_frames(w, h, 1 + 5 * 2, seed=7)
    p = params(3, occlusion_reasoning=1)
    whole = jets(ctx, frames, p, 3)
    a = jets(ctx, frames, p, 2, first_jet=0)
    b = jets(ctx, frames, p, 1, first_jet=2)
    joined = dict(params=b["params"], fwd=a["fwd"] + b["fwd"], back=a["back"] + b["back"], occ=a["occ"] + b["occ"],
                  outer=a["outer"] + b["outer"])
    assert_equal(joined, whole)
    assert_equal(b, composition(ctx, frames, p, 1, first_jet=2))


def frame_ints(frames):
    fa = (FrameInt * len(frames))()
    for k, f in enumerate(frames):
        fa[k] = FrameInt(f.shape[1], f.shape[0], 1 if f.ndim == 2 else f.shape[2], f.strides[0], f.ctypes.data)
    return fa


def sentinel_planes(w, h, n_jets, buffers=None):
    """fwd_x, fwd_y, back_x, back_y, occlusions: n_jets sentinel-filled planes each (buffers: a factory of float32 arrays)"""
    planes = [[Image(w, h, None if buffers is None else buffers(ceil4(w) * h)) for _ in range(n_jets)] for _ in range(5)]
    for ps in planes:
        for x in ps:
            x.buf[:] = SENTINEL
    return planes


def call(ctx, fa, bits, p, n_jets, planes, first_jet=0, scale=1.0, null=None):
    """the C entry on sentinel planes; null: index of an output array passed as NULL"""
    arrays = [(IP * max(len(ps), 1))(*[C.pointer(x.c) for x in ps]) for ps in planes]
    if null is not None:
        arrays[null] = None
    return ctx.lib.sfgpu_slow_flow_jets(ctx.h, len(fa), fa, bits, scale, first_jet, n_jets, C.byref(p), 0, None, *arrays)


@contextlib.contextmanager
def registered(ctx, bufs):
    done = []
    try:
        for b in bufs:
            assert ctx.lib.sfgpu_host_register(b.ctypes.data, b.nbytes) == 0
            done.append(b)
        yield
    finally:
        for b in done:
            ctx.lib.sfgpu_host_unregister(b.ctypes.data)


def test_jets_page_locked_equals_pageable(ctx):
    """Five jets reach every wait of the copy pipeline (frames of jet k + 1 behind the conversions of jet k, download
    planes of jet k behind the drain of jet k - 2) and reuse the event rings."""
    w, h = 200, 120
    frames = int_frames(w, h, 1 + 7 * 2, seed=3)
    p = params(3, occlusion_reasoning=1)
    pageable = sentinel_planes(w, h, 5)
    assert call(ctx, frame_ints(frames), 8, clone(p), 5, pageable) == 0
    kept = []

    def buffers(n):
        kept.append(own_pages((n,), np.float32))
        return kept[-1]

    locked = sentinel_planes(w, h, 5, buffers)
    with registered(ctx, frames + kept):  # contiguous (no row padding), each on its own pages
        assert call(ctx, frame_ints(frames), 8, clone(p), 5, locked) == 0
    for a, b in zip(pageable, locked):
        for x, y in zip(a, b):
            assert same(x.buf, y.buf)
    want = composition(ctx, frames, p, 5)
    for k in range(5):
        assert same(locked[0][k].buf, want["fwd"][k][0]) and same(locked[3][k].buf, want["back"][k][1])
        assert same(locked[4][k].buf, want["occ"][k])


def test_jets_argument_errors_write_nothing(ctx):
    w, h = 40, 32
    p = params(2)
    f8, f16 = int_frames(w, h, 5), int_frames(w, h, 5, np.uint16, top=1000)

    def fields(frames, k=None, **kw):
        fa = frame_ints(frames)
        for name, v in kw.items():
            setattr(fa[k], name, v)
        return fa

    cases = [
        ("bits", fields(f8), 12, {}),
        ("too few frames", fields(f8[:4]), 8, {}),
        ("frame size", fields(f8, 3, width=w - 4), 8, {}),
        ("frame channels", fields(f8, 1, channels=2), 8, {}),
        ("frame step too short", fields(f16, 2, step=3 * w * 2 - 2), 16, {}),
        ("frame step odd", fields(f16, 2, step=3 * w * 2 + 1), 16, {}),
        ("output geometry", fields(f8), 8, dict(out=(w + 1, h))),
        ("null output array", fields(f8), 8, dict(null=2)),
        ("n_jets", fields(f8), 8, dict(n_jets=0)),
        ("first_jet", fields(f8), 8, dict(first_jet=-1)),
        ("scale", fields(f8), 8, dict(scale=0.0)),
    ]
    for what, fa, bits, kw in cases:
        q = clone(p)
        ow, oh = kw.pop("out", (w, h))
        n_jets = kw.pop("n_jets", 2)
        planes = sentinel_planes(ow, oh, max(n_jets, 1))
        assert call(ctx, fa, bits, q, n_jets, planes, **kw) == 2, what
        assert all((x.buf == SENTINEL).all() for ps in planes for x in ps), what
        assert bytes(q) == bytes(p), what
    q = clone(p)
    q.smoothing = 2
    planes = sentinel_planes(w, h, 2)
    assert call(ctx, frame_ints(f8), 8, q, 2, planes) == 4
    assert all((x.buf == SENTINEL).all() for ps in planes for x in ps)
