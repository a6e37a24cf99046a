"""sfgpu_slow_flow_jets_epic against the composition it replaces, built from the existing entries: integer frame -> float32
-> ctx.prescale (scale != 1) -> ctx.normalize over all frames, then per window ctx.rgb_to_lab of its normalised reference
frame (saliency filter on) -> ctx.epic on a fresh copy of the edge map -> x 1/(S-1) in float32 -> Variational_MT -> x (S-1)
in float32.  Every output plane is compared bit for bit, stride padding included, together with the EPIC stats, the
published img_norm_* and the edge maps the call leaves behind (the originals + euc, added once)."""
import ctypes as C

import numpy as np
import pytest

import test_gpu_slow_flow_jets as sj
from slowflow_b200 import ColorImage, Image, Variational_MT, synth
from slowflow_b200.api import EpicStats, FloatImage, epic_params_default
from slowflow_b200.image import ceil4, image_t

pytestmark = pytest.mark.gpu

SENTINEL = sj.SENTINEL
FIP = C.POINTER(FloatImage)


def epic_inputs(w, h, steps, n_jets, counts=(300,), seed=1):
    """Matches of every window (the texture moves 0.7 x gt_flow per frame: 0.7 x steps to the reference frame's
    neighbours, with noise and a few outliers for the consistency filter) and n_jets + 1 edge maps, all in the window
    geometry w x h.  counts: match counts, cycled over the windows."""
    rng = np.random.RandomState(seed)
    u, v = synth.gt_flow(w, h)
    fwd, back, it = [], [], 0
    for _ in range(n_jets):
        for sign, out in ((1.0, fwd), (-1.0, back)):
            n = counts[it % len(counts)]
            it += 1
            xs, ys = rng.randint(1, w - 1, n), rng.randint(1, h - 1, n)
            m = np.zeros((n, 4), np.float32)
            m[:, 0], m[:, 1] = xs, ys
            m[:, 2] = xs + sign * 0.7 * steps * u[ys, xs] + rng.uniform(-0.3, 0.3, n)
            m[:, 3] = ys + sign * 0.7 * steps * v[ys, xs] + rng.uniform(-0.3, 0.3, n)
            bad = rng.rand(n) < 0.05
            m[bad, 2] += rng.uniform(-15, 15, int(bad.sum()))
            out.append(m)
    x = np.arange(w)[None, :]
    edges = [np.ascontiguousarray((0.1 + 0.8 * np.exp(-0.5 * ((x - w * (0.3 + 0.05 * i)) / 1.5) ** 2) +
                                   0.05 * rng.rand(h, w)).astype(np.float32)) for i in range(n_jets + 1)]
    return fwd, back, edges


def eparams(method="LA", filters=True):
    p = epic_params_default()
    p.method = method.encode()
    p.nn = 30
    if not filters:
        p.saliency_th, p.pref_nn = 0.0, 0
    return p


def normalised(ctx, frames, p, scale):
    ims = []
    for f in frames:
        a = f.astype(np.float32)
        a = np.stack([a] * 3) if a.ndim == 2 else np.moveaxis(a, 2, 0)
        im = ColorImage.from_array(a)
        ims.append(ctx.prescale(im, scale) if scale != 1.0 else im)
    q = sj.clone(p)
    ctx.normalize(ims, q)
    return ims, q


def composition(ctx, frames, p, n_jets, fwd_m, back_m, edges, ep, first_jet=0, scale=1.0, back_one=False, channel_w=None):
    """edges: the ORIGINAL maps (every sfgpu_epic call gets a fresh copy)"""
    steps = p.S - 1
    ims, q = normalised(ctx, frames, p, scale)
    w, h = ims[0].width, ims[0].height
    inv = np.float32(1) / np.float32(steps)
    out = dict(params=q, fwd=[], back=[], occ=[], stats=[])
    for k in range(n_jets):
        b = (first_jet + k) * steps
        for back in (False, True):
            ref = ims[b + 2 * steps] if back else ims[b + steps]
            lab = ctx.rgb_to_lab(ref) if ep.saliency_th != 0 else ref
            fx, fy = Image(w, h), Image(w, h)
            out["stats"].append(ctx.epic(fx, fy, lab, (back_m if back else fwd_m)[k], edges[k + back].copy(), ep))
            fx.buf[:] = fx.buf * inv
            fy.buf[:] = fy.buf * inv
            m = Variational_MT(ctx)
            if back:
                m.one_direction = back_one
                m.variational(fx, fy, [ims[b + 3 * steps - i] for i in range(2 * steps + 1)], q)
            else:
                m.setChannelWeights(channel_w)
                m.variational(fx, fy, ims[b:b + 2 * steps + 1], q)
                out["occ"].append(m.getOcclusions().buf.copy())
            out["back" if back else "fwd"].append((fx.buf * np.float32(steps), fy.buf * np.float32(steps)))
    return out


def jets_epic(ctx, frames, p, n_jets, fwd_m, back_m, edges, ep, **kw):
    q = sj.clone(p)
    fwd, back, occ, stats = ctx.slow_flow_jets_epic(frames, q, n_jets, fwd_m, back_m, edges, ep, occlusions=True, **kw)
    return dict(params=q, fwd=[(x.buf, y.buf) for x, y in fwd], back=[(x.buf, y.buf) for x, y in back], occ=[o.buf for o in occ],
                stats=stats)


def stats_tuple(s):
    return tuple(getattr(s, f) for f, _ in EpicStats._fields_)


def assert_equal(got, want):
    sj.assert_equal(got, want, outer=False)
    assert [stats_tuple(s) for s in got["stats"]] == [stats_tuple(s) for s in want["stats"]]


CASES = {
    "u8_rgb_S2_occlusions_LA": dict(shape=(96, 64), S=2, n_jets=1, kw=dict(occlusion_reasoning=1)),
    "u16_padded_step_S3_hbit_four_jets": dict(shape=(96, 64), S=3, n_jets=4, dtype=np.uint16, top=4095, pad=3, kw=dict(hbit=1)),
    "u8_grey_odd_width_five_jets": dict(shape=(77, 61), S=2, n_jets=5, channels=1),
    "scale_half": dict(shape=(130, 100), S=2, n_jets=2, scale=0.5),
    "two_layers": dict(shape=(96, 64), S=2, n_jets=2, kw=dict(layers=2, p_scale=0.8)),
    "backward_one_direction": dict(shape=(96, 64), S=2, n_jets=2, back_one=True),
    "NW": dict(shape=(96, 64), S=2, n_jets=2, method="NW"),
    "filters_off_no_lab": dict(shape=(96, 64), S=2, n_jets=2, filters=False),
    "mixed_match_counts": dict(shape=(96, 64), S=2, n_jets=3, counts=(300, 40, 170, 60, 80)),
    "nine_jets_first_jet_2": dict(shape=(80, 48), S=2, n_jets=9, first_jet=2),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_jets_epic_equal_composition(ctx, name):
    c = CASES[name]
    w, h = c["shape"]
    steps = c["S"] - 1
    first, n_jets, scale = c.get("first_jet", 0), c["n_jets"], c.get("scale", 1.0)
    frames = sj.int_frames(w, h, 1 + (first + n_jets + 2) * steps, c.get("dtype", np.uint8), c.get("channels", 3), c.get("top", 255),
                           c.get("pad", 0))
    p = sj.params(c["S"], **c.get("kw", {}))
    ww, hh = (round(w * scale), round(h * scale)) if scale != 1.0 else (w, h)
    fwd_m, back_m, edges = epic_inputs(ww, hh, steps, n_jets, c.get("counts", (300,)))
    ep = eparams(c.get("method", "LA"), c.get("filters", True))
    back_one = c.get("back_one", False)
    want = composition(ctx, frames, p, n_jets, fwd_m, back_m, edges, ep, first, scale, back_one)
    mine = [e.copy() for e in edges]
    got = jets_epic(ctx, frames, p, n_jets, fwd_m, back_m, mine, ep, first_jet=first, scale=scale, backward_one_direction=back_one)
    if scale != 1.0:
        assert got["fwd"][0][0].size == ceil4(ww) * hh
    assert all(np.isfinite(x).all() for f in got["fwd"] + got["back"] for x in f)
    assert all(s.matches_after_consistency > 0 for s in got["stats"])
    assert_equal(got, want)
    for e, m in zip(edges, mine):  # euc added once to every map
        assert sj.same(m, e + np.float32(ep.euc))


def test_jets_epic_channel_weights(ctx):
    w, h = 96, 64
    frames = sj.int_frames(w, h, 6, seed=11)
    cw = ColorImage(w, h)
    cw.buf[:] = 1.0
    ctx.raw_weighting(cw, 1, 0, 2.0)
    p = sj.params(2)
    fwd_m, back_m, edges = epic_inputs(w, h, 1, 2, seed=4)
    ep = eparams()
    want = composition(ctx, frames, p, 2, fwd_m, back_m, edges, ep, channel_w=cw)
    assert_equal(jets_epic(ctx, frames, p, 2, fwd_m, back_m, [e.copy() for e in edges], ep, channel_w=cw), want)


def float_images(arrays):
    fis = [FloatImage(a.ctypes.data_as(C.POINTER(C.c_float)), a.shape[1], a.shape[0]) for a in arrays]
    return fis, (FIP * max(len(fis), 1))(*[C.pointer(x) for x in fis])


def call(ctx, fa, bits, p, n_jets, planes, fwd_m, back_m, edges, ep, stats=None, first_jet=0, edge_structs=None):
    """the C entry on sentinel planes; edge_structs: a ready float_image* array instead of one made from `edges`"""
    IP = C.POINTER(image_t)
    arrays = [(IP * max(len(ps), 1))(*[C.pointer(x.c) for x in ps]) for ps in planes]
    fm, bm = float_images(fwd_m), float_images(back_m)
    ed = float_images(edges) if edge_structs is None else (None, edge_structs)
    return ctx.lib.sfgpu_slow_flow_jets_epic(ctx.h, len(fa), fa, bits, 1.0, first_jet, n_jets, C.byref(p), 0, None, fm[1], bm[1], ed[1],
                                             None if ep is None else C.byref(ep), *arrays, stats)


def test_jets_epic_page_locked_equals_pageable(ctx):
    """Nine jets: three chunks, so every wait of the copy pipeline (next chunk's frames and edge maps behind this chunk's
    EPIC batch, download planes behind the drain of jet k - 2) is reached and the event rings are reused."""
    w, h, n = 120, 80, 9
    frames = sj.int_frames(w, h, 1 + (n + 2) * 2, seed=3)
    p = sj.params(3, occlusion_reasoning=1)
    fwd_m, back_m, edges = epic_inputs(w, h, 2, n, seed=8)
    ep = eparams()
    pageable = sj.sentinel_planes(w, h, n)
    e1 = [e.copy() for e in edges]
    st1 = (EpicStats * (2 * n))()
    assert call(ctx, sj.frame_ints(frames), 8, sj.clone(p), n, pageable, fwd_m, back_m, e1, ep, st1) == 0, ctx.lib.sfgpu_last_error()
    kept = []

    def buffers(k):
        kept.append(sj.own_pages((k,), np.float32))
        return kept[-1]

    locked = sj.sentinel_planes(w, h, n, buffers)
    e2 = []
    for e in edges:
        e2.append(sj.own_pages(e.shape, np.float32))
        e2[-1][:] = e
    st2 = (EpicStats * (2 * n))()
    with sj.registered(ctx, frames + kept + e2):
        assert call(ctx, sj.frame_ints(frames), 8, sj.clone(p), n, locked, fwd_m, back_m, e2, ep, st2) == 0, ctx.lib.sfgpu_last_error()
    for a, b in zip(pageable, locked):
        for x, y in zip(a, b):
            assert sj.same(x.buf, y.buf)
    assert [stats_tuple(s) for s in st1] == [stats_tuple(s) for s in st2]
    for a, b in zip(e1, e2):
        assert sj.same(a, b)
    want = composition(ctx, frames, p, n, fwd_m, back_m, edges, ep)
    for k in range(n):
        assert sj.same(locked[0][k].buf, want["fwd"][k][0]) and sj.same(locked[1][k].buf, want["fwd"][k][1])
        assert sj.same(locked[2][k].buf, want["back"][k][0]) and sj.same(locked[3][k].buf, want["back"][k][1])
        assert sj.same(locked[4][k].buf, want["occ"][k])
    assert [stats_tuple(s) for s in st2] == [stats_tuple(s) for s in want["stats"]]


def test_jets_epic_no_match_stops_at_its_chunk(ctx):
    """Jet 5's backward window has no match: chunk 0 (jets 0-3) is complete, jets 4-8 are not written, the edge maps of
    chunks 0 and 1 carry euc and the last one (chunk 2's) is untouched."""
    w, h, n = 80, 48, 9
    frames = sj.int_frames(w, h, 1 + (n + 2), seed=9)
    p = sj.params(2)
    fwd_m, back_m, edges = epic_inputs(w, h, 1, n, seed=12)
    back_m[5] = np.zeros((1, 4), np.float32)[:0]  # no rows, non-null data
    ep = eparams(filters=False)
    planes = sj.sentinel_planes(w, h, n)
    mine = [e.copy() for e in edges]
    st = (EpicStats * (2 * n))()
    assert call(ctx, sj.frame_ints(frames), 8, sj.clone(p), n, planes, fwd_m, back_m, mine, ep, st) == 2
    msg = ctx.lib.sfgpu_last_error().decode()
    assert "jet 5 backward" in msg and "no match" in msg, msg
    want = composition(ctx, frames, p, 4, fwd_m, back_m, edges, ep)
    for k in range(4):
        assert sj.same(planes[0][k].buf, want["fwd"][k][0]) and sj.same(planes[3][k].buf, want["back"][k][1])
        assert sj.same(planes[4][k].buf, want["occ"][k])
    assert [stats_tuple(s) for s in st[:8]] == [stats_tuple(s) for s in want["stats"]]
    assert all(stats_tuple(s) == (0,) * 5 for s in st[8:])
    assert all((x.buf == SENTINEL).all() for ps in planes for x in ps[4:])
    for i in range(n):
        assert sj.same(mine[i], edges[i] + np.float32(ep.euc)), i
    assert sj.same(mine[n], edges[n])


def test_jets_epic_argument_errors_touch_nothing(ctx):
    w, h, n = 40, 32, 2
    p = sj.params(2)
    frames = sj.int_frames(w, h, 5)
    fwd_m, back_m, edges = epic_inputs(w, h, 1, n)
    ep = eparams()
    bad_method = eparams()
    bad_method.method = b"XX"
    three_cols = [np.ascontiguousarray(m[:, :3]) for m in fwd_m]
    small = [e[:-1].copy() for e in edges]
    cases = [
        ("too few frames", dict(frames=frames[:4])),
        ("match columns", dict(fwd_m=three_cols)),
        ("edge geometry", dict(edges=small)),
        ("method", dict(ep=bad_method)),
        ("null epic_params", dict(ep=None)),
        ("shared edge array", dict(share=True)),
        ("output geometry", dict(out=(w + 1, h))),
    ]
    for what, kw in cases:
        mine = [e.copy() for e in kw.get("edges", edges)]
        edge_structs = None
        if kw.get("share"):
            fis, edge_structs = float_images(mine)
            edge_structs[2] = edge_structs[0]
        ow, oh = kw.get("out", (w, h))
        planes = sj.sentinel_planes(ow, oh, n)
        q = sj.clone(p)
        st = (EpicStats * (2 * n))()
        rc = call(ctx, sj.frame_ints(kw.get("frames", frames)), 8, q, n, planes, kw.get("fwd_m", fwd_m), back_m, mine, kw.get("ep", ep), st,
                  edge_structs=edge_structs)
        assert rc == 2, what
        assert all((x.buf == SENTINEL).all() for ps in planes for x in ps), what
        assert all(sj.same(a, b) for a, b in zip(mine, kw.get("edges", edges))), what
        assert bytes(q) == bytes(p), what
        assert all(stats_tuple(s) == (0,) * 5 for s in st), what
    q = sj.clone(p)
    q.smoothing = 2
    planes = sj.sentinel_planes(w, h, n)
    mine = [e.copy() for e in edges]
    assert call(ctx, sj.frame_ints(frames), 8, q, n, planes, fwd_m, back_m, mine, ep) == 4
    assert all((x.buf == SENTINEL).all() for ps in planes for x in ps)
    assert all(sj.same(a, b) for a, b in zip(mine, edges))


def test_slow_flow_jets_after_epic_call(ctx):
    """sfgpu_slow_flow_jets on a context the EPIC variant has used (larger ring, EPIC arena) still equals its composition."""
    w, h = 96, 64
    frames = sj.int_frames(w, h, 1 + 6 * 2, seed=21)
    p = sj.params(3, occlusion_reasoning=1)
    fwd_m, back_m, edges = epic_inputs(w, h, 2, 4, seed=2)
    jets_epic(ctx, frames, p, 4, fwd_m, back_m, edges, eparams())
    sj.assert_equal(sj.jets(ctx, frames, p, 4), sj.composition(ctx, frames, p, 4))
