"""The default two-frame loop runs one data pass per outer iteration (k_prep_fused: flow update, smoothness
diffusivities, warp, derivatives, data term, Laplacian and block inverse).  SLOWFLOW_GPU_DATA_VARIANT=2 keeps the
smoothness pass separate (k_flow_smooth + k_prep_two_frame).  The two must give the same flow bit for bit, padding
columns included."""
import numpy as np
import pytest

import helpers
from slowflow_b200 import Context, Image, synth, variational_params_default

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("built")]


def _params(niter_outer=5, delta=0.0):
    p = variational_params_default()
    p.niter_outer = niter_outer
    p.delta = delta
    return p


def _case(w, h, leaving=False, seed=20170721):
    """Seeded frame pair and initial flow; the padding columns of the flow hold arbitrary finite values (the flow update
    stores w + du there).  leaving: a flow that points out of the image on all four sides."""
    im1, im2, wx, wy = helpers.pair(w, h, seed)
    if leaving:
        y, x = np.mgrid[0:h, 0:w].astype(np.float32)
        wx.array[:] += 0.08 * (x - 0.5 * w)
        wy.array[:] += 0.08 * (y - 0.5 * h)
    r = np.random.RandomState(seed + 1)
    pad = wx.stride - w
    if pad:
        wx.full[:, w:] = r.uniform(-3, 3, size=(h, pad)).astype(np.float32)
        wy.full[:, w:] = r.uniform(-3, 3, size=(h, pad)).astype(np.float32)
    return im1, im2, wx, wy


def _same(a, b):
    return np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _both_variants(monkeypatch, run):
    with Context(0) as c0:
        a = run(c0)
    monkeypatch.setenv("SLOWFLOW_GPU_DATA_VARIANT", "2")
    with Context(0) as c2:
        b = run(c2)
    return a, b


@pytest.mark.parametrize("w,h,niter_outer,delta,leaving", [
    (61, 45, 5, 0.0, False),
    (61, 45, 1, 0.5, True),
    (333, 211, 5, 0.0, True),   # stride != width
    (333, 211, 1, 0.0, False),
    (237, 90, 5, 0.5, False),   # 3 padding columns, colour term
    (254, 77, 5, 0.0, True),    # 2 padding columns
    (255, 64, 5, 0.5, True),    # 1 padding column
    (2073, 1166, 5, 0.0, True),
    (2560, 1440, 5, 0.0, False),
    (2560, 1440, 5, 0.5, True),
])
def test_fused_data_pass_matches_separate_smoothness_pass(monkeypatch, w, h, niter_outer, delta, leaving):
    im1, im2, wx0, wy0 = _case(w, h, leaving)
    p = _params(niter_outer, delta)

    def run(c):
        a, b = wx0.copy(), wy0.copy()
        c.variational(a, b, im1, im2, p)
        return a.buf.copy(), b.buf.copy()

    (ax, ay), (bx, by) = _both_variants(monkeypatch, run)
    assert np.isfinite(ax).all() and np.isfinite(ay).all()
    assert _same(ax, bx) and _same(ay, by)
    # the flow moved: the comparison is not between two untouched copies of the input
    assert not _same(ax, wx0.buf)


def test_fused_data_pass_device_entry(monkeypatch):
    torch = pytest.importorskip("torch")
    w, h = 1021, 333
    im1, im2, wx0, wy0 = _case(w, h, leaving=True)
    p = _params(5, 0.25)

    def run(c):
        t = lambda x: torch.from_numpy(x.buf.copy()).cuda()
        d1, d2, dx, dy = t(im1), t(im2), t(wx0), t(wy0)
        torch.cuda.synchronize()
        c.variational_dev(dx.data_ptr(), dy.data_ptr(), d1.data_ptr(), d2.data_ptr(), w, h, wx0.stride, p)
        c.synchronize()
        return dx.cpu().numpy(), dy.cpu().numpy()

    (ax, ay), (bx, by) = _both_variants(monkeypatch, run)
    assert _same(ax, bx) and _same(ay, by)


def test_fused_data_pass_integer_sequence(monkeypatch):
    w, h, n = 322, 200, 3
    raws = [np.ascontiguousarray(np.moveaxis(np.rint(synth.frame(w, h, t)).clip(0, 255).astype(np.uint8), 0, 2))
            for t in range(n + 1)]
    u0, v0 = synth.initial_flow(w, h)

    def run(c):
        xs, ys = [Image.from_array(u0) for _ in range(n)], [Image.from_array(v0) for _ in range(n)]
        c.variational_sequence_int(raws, xs, ys, None)
        return [x.buf.copy() for x in xs], [y.buf.copy() for y in ys]

    (ax, ay), (bx, by) = _both_variants(monkeypatch, run)
    for j in range(n):
        assert _same(ax[j], bx[j]) and _same(ay[j], by[j]), j
