"""The copy pipeline of the sequence entries (CopyPipeline, slowflow_b200/csrc/sf_hostcopy.cu) with page-locked caller memory.

With registered buffers, uploads and downloads run on their own streams, ordered by rings of 4 events per kind.  Seven
pairs reach every wait the sequence uses ("compute passed pair j-2", "drained pair j-3") and reuse every ring slot.  Each
case is compared bit for bit with a path that orders its copies differently: pageable buffers (every copy on the compute
stream), single-pair calls, the float sequence, or the per-pair EpicFlow composition."""
import contextlib
import mmap

import numpy as np
import pytest

from slowflow_b200 import ColorImage, Image, synth, variational_params_default
from slowflow_b200.api import epic_params_default

pytestmark = pytest.mark.gpu

N_PAIRS = 7
SENTINEL = np.float32(-12345.5)


@pytest.fixture(scope="module")
def ctx(built):
    from slowflow_b200 import Context
    c = Context(0)
    yield c
    c.close()


def own_pages(shape, dtype=np.float32):
    """A zeroed array on pages no other array uses, so that registering it never overlaps another registration."""
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    raw = np.zeros(nbytes + 2 * mmap.PAGESIZE, np.uint8)
    off = (-raw.ctypes.data) % mmap.PAGESIZE
    return raw[off:off + nbytes].view(dtype).reshape(shape)


def image(a):
    h, w = a.shape
    im = Image(w, h, own_pages(((w + 3) // 4 * 4) * h))
    im.array[:] = a
    return im


def color_image(a):
    _, h, w = a.shape
    im = ColorImage(w, h, own_pages(3 * ((w + 3) // 4 * 4) * h))
    im.array[:] = a
    return im


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


def flows(u0, v0, n=N_PAIRS):
    return [image(u0) for _ in range(n)], [image(v0) for _ in range(n)]


def assert_same(ax, ay, bx, by):
    assert len(ax) == len(bx)
    for j in range(len(ax)):
        for name, a, b in (("wx", ax[j].buf, bx[j].buf), ("wy", ay[j].buf, by[j].buf)):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), "pair %d: %s differs at %d entries" % (
                j, name, int((a.view(np.uint32) != b.view(np.uint32)).sum()))


@pytest.fixture(scope="module")
def float_case(ctx):
    """1024x600 (flow planes of 2.4 MB: above the staging threshold), 7 pairs, and the sequence on pageable buffers."""
    w, h = 1024, 600
    frames = [color_image(synth.frame(w, h, t)) for t in range(N_PAIRS + 1)]
    u0, v0 = synth.initial_flow(w, h)
    px, py = flows(u0, v0)
    ctx.variational_sequence(frames, px, py, None)  # nothing registered: the pageable path
    return frames, u0, v0, px, py


def test_registered_sequence_equals_pageable_and_single_pairs(ctx, float_case):
    frames, u0, v0, px, py = float_case
    rx, ry = flows(u0, v0)
    with registered(ctx, [f.buf for f in frames] + [p.buf for p in rx + ry]):
        ctx.variational_sequence(frames, rx, ry, None)
    assert_same(rx, ry, px, py)
    sx, sy = flows(u0, v0)
    for j in range(N_PAIRS):
        ctx.variational(sx[j], sy[j], frames[j], frames[j + 1], None)
    assert_same(rx, ry, sx, sy)


def test_one_pageable_flow_plane_takes_the_pageable_path(ctx, float_case):
    frames, u0, v0, px, py = float_case
    mx, my = flows(u0, v0)
    with registered(ctx, [f.buf for f in frames] + [p.buf for p in mx] + [p.buf for k, p in enumerate(my) if k != 3]):
        ctx.variational_sequence(frames, mx, my, None)
    assert_same(mx, my, px, py)


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_registered_integer_sequence_equals_float_sequence(ctx, dtype):
    """3-channel frames with a row step > width * channels.  16-bit frames hold 10-bit data: full-range 16-bit intensities
    drive the two-frame smoothness weight exp(-5 |grad lum / 255|) to 0 and the reference itself to NaN."""
    w, h = 322, 200
    top = 255 if dtype == np.uint8 else 1020
    canvases, floats = [], []
    for t in range(N_PAIRS + 1):
        f = np.rint(synth.frame(w, h, t) * (top / 255.0)).astype(dtype)  # (3, H, W)
        canvas = own_pages((h, w + 5, 3), dtype)
        canvas[:, :w, :] = np.moveaxis(f, 0, 2)
        canvases.append(canvas)
        floats.append(color_image(f.astype(np.float32)))
    raws = [c[:, :w, :] for c in canvases]
    u0, v0 = synth.initial_flow(w, h)
    params = variational_params_default()
    ax, ay = flows(u0, v0)
    ctx.variational_sequence(floats, ax, ay, params)
    bx, by = flows(u0, v0)
    cx, cy = flows(u0, v0)
    with registered(ctx, canvases + [p.buf for p in bx + by + cx + cy]):
        ctx.variational_sequence_int(raws, bx, by, params)
        # the same run in two calls, the second continuing from the frame the first one left on the device
        ctx.variational_sequence_int(raws[:4], cx[:3], cy[:3], params)
        ctx.variational_sequence_int(raws[3:], cx[3:], cy[3:], params, continue_from_previous=True)
    assert all(np.isfinite(x.array).all() for x in ax)
    assert_same(bx, by, ax, ay)
    assert_same(cx, cy, ax, ay)


def test_registered_epicflow_pair_without_matches_stops_at_its_chunk(ctx):
    """Pair 9 of 19 (chunk 1) has a flat first frame, so the saliency filter removes every match.  With page-locked
    buffers chunk 0 is complete and equals the composition, pairs 8..18 keep their planes and chunk 2's edge maps are
    untouched."""
    w, h, n = 160, 120, 19
    frames = [color_image(synth.frame(w, h, t, 700)) for t in range(n + 1)]
    frames[9] = color_image(np.zeros((3, h, w), np.float32))
    ms, es = [], []
    for k in range(n):
        _, m, e = synth.epic_case(w, h, 300, seed=700 + 31 * k)
        ms.append(m)
        es.append(np.clip(e + 0.05 * np.random.RandomState(700 + k).rand(h, w), 0.0, 1.0).astype(np.float32))
    ep = epic_params_default()

    def sentinel_planes(count):
        out = [(image(np.zeros((h, w), np.float32)), image(np.zeros((h, w), np.float32))) for _ in range(count)]
        for fx, fy in out:
            fx.buf[:], fy.buf[:] = SENTINEL, SENTINEL
        return out

    want, want_e = sentinel_planes(8), [e.copy() for e in es[:8]]
    for k, (fx, fy) in enumerate(want):  # rgb_to_lab -> epic -> variational, pair by pair
        ctx.epic(fx, fy, ctx.rgb_to_lab(frames[k]), ms[k], want_e[k], ep)
        ctx.variational(fx, fy, frames[k], frames[k + 1], None)
    fl = sentinel_planes(n)
    eo = []
    for e in es:
        eo.append(own_pages(e.shape))
        eo[-1][:] = e
    with registered(ctx, [f.buf for f in frames] + [p.buf for f in fl for p in f] + eo):
        with pytest.raises(RuntimeError, match=r"status 2\).*pair 9: no match survived the filters"):
            ctx.epicflow_sequence(frames, ms, eo, [f[0] for f in fl], [f[1] for f in fl], ep)
    assert_same([f[0] for f in fl[:8]], [f[1] for f in fl[:8]], [f[0] for f in want], [f[1] for f in want])
    for k in range(8):
        assert np.array_equal(eo[k].view(np.uint32), want_e[k].view(np.uint32)), "pair %d: edges" % k
    assert all((fx.buf == SENTINEL).all() and (fy.buf == SENTINEL).all() for fx, fy in fl[8:])
    assert all(np.array_equal(eo[k], es[k]) for k in range(16, n))
