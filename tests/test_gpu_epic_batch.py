"""sfgpu_epic_batch: EPIC on n images of one geometry in one call (slowflow_b200/csrc/sf_epic.cu).  Every item must equal its
own sfgpu_epic call bit for bit: whole flow planes (padding included), the five stats, and the edge map after += euc.

The items differ in their matches (synth.epic_case with a seed per item) and in a seeded perturbation of the edge costs, so
that their label maps, match counts and sweep counts differ."""
import ctypes as C
import threading

import numpy as np
import pytest

import epic_helpers as eh
from slowflow_b200 import ColorImage, Image, synth
from slowflow_b200.api import EpicStats, FloatImage, epic_params_default
from slowflow_b200.image import color_image_t, image_t

pytestmark = pytest.mark.gpu

SENTINEL = np.float32(-12345.5)  # what the flow planes hold before a call (padding included)
STATS = ("matches_in", "matches_after_saliency", "matches_after_consistency", "sweeps_prefilter", "sweeps_interpolation")


def params(method="LA", filters=True):
    p = epic_params_default()
    p.method = method.encode()
    if not filters:
        p.saliency_th, p.pref_nn = 0.0, 0
    return p


def item(w, h, n, seed, filters=True):
    """-> (image, matches, edges) of one batch item."""
    im, m, edges = synth.epic_case(w, h, n, seed=seed, outliers=0.05 if filters else 0.0)
    edges = np.clip(edges + 0.05 * np.random.RandomState(seed).rand(h, w), 0.0, 1.0).astype(np.float32)
    return ColorImage.from_array(im), m, edges


def planes(w, h, n):
    out = []
    for _ in range(n):
        fx, fy = Image(w, h), Image(w, h)
        fx.buf[:], fy.buf[:] = SENTINEL, SENTINEL
        out.append((fx, fy))
    return out


def run_single(ctx, items, p, w, h):
    fl, es, st = planes(w, h, len(items)), [], []
    for (im, m, e), (fx, fy) in zip(items, fl):
        e = e.copy()
        st.append(ctx.epic(fx, fy, im, m, e, p))
        es.append(e)
    return fl, es, st


def run_batch(ctx, items, p, w, h):
    fl, es = planes(w, h, len(items)), [e.copy() for _, _, e in items]
    st = ctx.epic_batch([f[0] for f in fl], [f[1] for f in fl], [i[0] for i in items], [i[1] for i in items], es, p)
    return fl, es, st


def assert_same(a, b):
    (fa, ea, sa), (fb, eb, sb) = a, b
    assert len(fa) == len(fb)
    for k in range(len(fa)):
        for name, x, y in (("flow x", fa[k][0].buf, fb[k][0].buf), ("flow y", fa[k][1].buf, fb[k][1].buf), ("edges", ea[k], eb[k])):
            assert np.array_equal(x.view(np.uint32), y.view(np.uint32)), "item %d: %s differs at %d entries" % (
                k, name, int((x.view(np.uint32) != y.view(np.uint32)).sum()))
        assert [getattr(sa[k], f) for f in STATS] == [getattr(sb[k], f) for f in STATS], "item %d: stats differ" % k


@pytest.mark.parametrize("w,h,counts,method,filters", [
    (320, 200, [800] * 5, "LA", True), (320, 200, [800] * 5, "NW", True), (320, 200, [800] * 5, "LA", False),
    (320, 200, [800] * 5, "NW", False),
    (501, 333, [2500] * 3, "LA", True),  # odd width: stride != width
    (1024, 436, [5000] * 8, "LA", True),
    # match counts per item: 20 and 90 leave fewer than nn = 100 (and 20 fewer than pref_nn + 1 = 26), so nns differs per item
    (320, 200, [800, 90, 1500, 20, 300], "LA", True), (320, 200, [800, 90, 1500, 20, 300], "NW", True),
    # strip-pipeline edge geometries: narrower than a 32-column block, five rows
    (31, 7, [12] * 4, "LA", False), (100, 5, [12] * 4, "LA", False), (31, 7, [12] * 4, "NW", False), (100, 5, [12] * 4, "NW", False),
])
def test_batch_equals_single_calls(ctx, w, h, counts, method, filters):
    items = [item(w, h, n, 500 + 31 * k, filters) for k, n in enumerate(counts)]
    p = params(method, filters)
    single, batch = run_single(ctx, items, p, w, h), run_batch(ctx, items, p, w, h)
    assert_same(batch, single)
    st = batch[2]
    print("%dx%d %s: consistency %s, sweeps %s" % (w, h, method, [s.matches_after_consistency for s in st],
                                                   [(s.sweeps_prefilter, s.sweeps_interpolation) for s in st]))
    assert all(s.matches_after_consistency > 0 for s in st)


def test_batch_beyond_one_resident_group(ctx):
    """2560x1440 has 45 strips of 32 rows; 14 items are 630 strips, more than 4 per SM on 148 SMs, so the distance transforms
    run in two groups."""
    w, h = 2560, 1440
    items = [item(w, h, 3000, 900 + k) for k in range(14)]
    p = params()
    assert_same(run_batch(ctx, items, p, w, h), run_single(ctx, items, p, w, h))


@pytest.mark.parametrize("w,h,n,method,filters", eh.REGRESSION_EPIC)
def test_batch_middle_item_unchanged_since_recorded(ctx, w, h, n, method, filters):
    """Each recorded EPIC case as the middle item of three still matches the regression vectors (the tolerance of
    test_epic_unchanged_since_recorded)."""
    g, t = np.load(eh.REGRESSION_FILE), eh.tag(w, h, n, method, filters)
    ci, m, edges, p = eh.epic_inputs(w, h, n, method, filters)
    items = [item(w, h, n, 77, filters), (ci, m, edges), item(w, h, n, 78, filters)]
    fl, es, st = run_batch(ctx, items, p, w, h)
    gx, gy = fl[1]
    assert [st[1].matches_in, st[1].matches_after_saliency, st[1].matches_after_consistency] == g["counts_" + t].tolist()
    assert np.array_equal(eh.stored(es[1], eh.FLOW_SAMPLE), g["edges_" + t])
    d = np.hypot(eh.stored(gx.array, eh.FLOW_SAMPLE) - g["fx_" + t], eh.stored(gy.array, eh.FLOW_SAMPLE) - g["fy_" + t])
    assert d.mean() <= 0.001 and d.max() <= 0.01, (d.mean(), d.max())


def raw_batch(ctx, n, fl, ims, ms, es, p):
    """sfgpu_epic_batch through ctypes, where an item of `fl` may be None (NULL flow planes) -> status."""
    IP, CP, FIP = C.POINTER(image_t), C.POINTER(color_image_t), C.POINTER(FloatImage)
    FP = C.POINTER(C.c_float)
    fm = [FloatImage(m.ctypes.data_as(FP), m.shape[1], m.shape[0]) for m in ms]
    fe = [FloatImage(e.ctypes.data_as(FP), e.shape[1], e.shape[0]) for e in es]
    k = len(fl)
    return ctx.lib.sfgpu_epic_batch(ctx.h, n, (IP * k)(*[C.pointer(f[0].c) if f else None for f in fl]),
                                    (IP * k)(*[C.pointer(f[1].c) if f else None for f in fl]), (CP * k)(*[C.pointer(i.c) for i in ims]),
                                    (FIP * k)(*[C.pointer(m) for m in fm]), (FIP * k)(*[C.pointer(e) for e in fe]), C.byref(p), (EpicStats * k)())


def untouched(fl):
    return all(f is None or ((f[0].buf == SENTINEL).all() and (f[1].buf == SENTINEL).all()) for f in fl)


def test_batch_errors_leave_flows_untouched(ctx):
    w, h = 160, 120
    items = [item(w, h, 300, 40 + k) for k in range(3)]
    p = params()
    ims, ms, es = [i[0] for i in items], [i[1] for i in items], [i[2].copy() for i in items]
    err = lambda: ctx.lib.sfgpu_last_error().decode()

    fl = planes(w, h, 3)
    assert raw_batch(ctx, 0, fl, ims, ms, es, p) == 2 and untouched(fl)

    fl = planes(w, h, 3)
    fl[1] = None  # a null item
    assert raw_batch(ctx, 3, fl, ims, ms, es, p) == 2 and untouched(fl)
    assert "item 1" in err()

    other = item(w, h + 1, 300, 43)  # items of different geometry
    fl = planes(w, h, 3)
    fl[2] = (Image(w, h + 1), Image(w, h + 1))
    fl[2][0].buf[:], fl[2][1].buf[:] = SENTINEL, SENTINEL
    assert raw_batch(ctx, 3, fl, [ims[0], ims[1], other[0]], ms[:2] + [other[1]], es[:2] + [other[2]], p) == 2 and untouched(fl)
    assert "item 2" in err() and "different geometry" in err()

    # item 2's image is flat: its saliency is 0 everywhere, so the saliency filter removes every match
    flat = ColorImage.from_array(np.zeros((3, h, w), np.float32))
    fl = planes(w, h, 3)
    with pytest.raises(RuntimeError, match=r"status 2\).*item 2: no match survived the filters"):
        ctx.epic_batch([f[0] for f in fl], [f[1] for f in fl], [ims[0], ims[1], flat], ms, [e.copy() for e in es], p)
    assert untouched(fl)


def test_concurrent_contexts_run_batches_like_sequential_runs(built):
    """Two host threads, each with its own context on cuda:0, run batches at the same time: their distance-transform launches
    (tickets and progress flags per context) share the SMs.  Results must equal the same batches run one after the other."""
    from slowflow_b200 import Context
    cases = [(320, 200, [800, 300, 1200, 800]), (1024, 436, [5000, 4000, 3000])]
    inputs = [[item(w, h, n, 1300 + 7 * i + k) for k, n in enumerate(counts)] for i, (w, h, counts) in enumerate(cases)]
    p = params()
    c0 = Context(0)
    ref = [run_batch(c0, inputs[i], p, w, h) for i, (w, h, _) in enumerate(cases)]
    c0.close()
    out, err = [None] * len(cases), []

    def work(i):
        try:
            c = Context(0)
            w, h, _ = cases[i]
            for _ in range(3):  # several calls per thread: the launches of the threads interleave differently each time
                r = run_batch(c, inputs[i], p, w, h)
                assert_same(r, ref[i])
            out[i] = r
            c.close()
        except Exception as e:  # pragma: no cover
            err.append(repr(e))

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(cases))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not err, err
    assert all(o is not None for o in out)
