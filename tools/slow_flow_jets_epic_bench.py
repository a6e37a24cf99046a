#!/usr/bin/env python3
"""The Slow Flow jet loop with EPIC initial flows: one sfgpu_slow_flow_jets_epic call against the strongest composition of
the existing entries.

Arms, run alternately in one process after one warm-up call of each per workload, with page-locked host buffers:
  (a) ctx.lib.sfgpu_slow_flow_jets_epic: integer frames and edge maps cross PCIe, everything else on the device, EPIC in
      batches of 8 windows, uploads and downloads overlapping the solves;
  (b) per chunk of 4 jets, as a caller builds it from the existing entries: the normalised float frames (host conversion +
      ctx.normalize over the whole sequence, once), ctx.rgb_to_lab of the chunk's normalised reference frames,
      ctx.epic_batch of its 8 windows, x 1/(S-1) on the host, then per window ctx.variational_mt with the frame cache on
      and x (S-1) on the host.
Each window of (b) gets its own copy of its reference frame's edge map (the reference reads the edge file per window);
the copies are refreshed outside the timed region.  Matches are synthetic: the ground-truth flow of the sequence x 0.7 x
(S-1) (the texture moves 0.7 x gt_flow per frame) plus uniform noise of +-0.3 px and 5 % outliers.
Every call ends with a stream synchronise, so a host clock around it measures the device work plus what the host adds.
The outputs of both arms (flows, occlusion labels, EPIC stats) are compared bit for bit on every repetition.  The card's
name, power limit and top SM clock are read in the same run.

    python tools/slow_flow_jets_epic_bench.py --out DIR [--reps 5] [--workloads NAME,...]
Writes DIR/slow_flow_jets_epic_bench.json and prints a summary.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import slow_flow_jets_bench as sjb  # noqa: E402  (device_info, parameters, frames, page-locking, summaries)

CHUNK = 4  # jets per EPIC batch of arm (b): the chunk of the one call
# name: (width, height, S, jets, parameter set, matches per window); the parameter sets of tools/slow_flow_jets_bench.py
WORKLOADS = {
    "1280x1024_u8": (1280, 1024, 3, 16, "driver", 5000),
    "2560x1440_config4_u8": (2560, 1440, 3, 4, "config4", 8000),
}


def parse():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="directory for slow_flow_jets_epic_bench.json")
    ap.add_argument("--reps", type=int, default=5, help="timed repetitions per arm and workload")
    ap.add_argument("--workloads", default=",".join(WORKLOADS), help="comma-separated subset of " + ", ".join(WORKLOADS))
    return ap.parse_args()


def epic_inputs(w, h, steps, jets, n, seed=5):
    """matches of every window (forward, backward per jet) and jets + 1 edge maps (SED-like: gradient magnitude of the
    texture's first frame plus the motion discontinuity at x = W/2)"""
    import numpy as np
    from slowflow_b200 import synth
    rng = np.random.RandomState(seed)
    u, v = synth.gt_flow(w, h)
    fwd, back = [], []
    for _ in range(jets):
        for sign, out in ((1.0, fwd), (-1.0, back)):
            xs, ys = rng.randint(2, w - 2, n), rng.randint(2, h - 2, n)
            m = np.zeros((n, 4), np.float32)
            m[:, 0], m[:, 1] = xs, ys
            m[:, 2] = xs + sign * 0.7 * steps * u[ys, xs] + rng.uniform(-0.3, 0.3, n)
            m[:, 3] = ys + sign * 0.7 * steps * v[ys, xs] + rng.uniform(-0.3, 0.3, n)
            bad = rng.rand(n) < 0.05
            m[bad, 2] += rng.uniform(-25, 25, int(bad.sum()))
            m[bad, 3] += rng.uniform(-25, 25, int(bad.sum()))
            out.append(m)
    _, _, e = synth.epic_case(w, h, 16)
    edges = [np.ascontiguousarray(e) for _ in range(jets + 1)]
    return fwd, back, edges


def float_images(arrays):
    from slowflow_b200.api import FloatImage
    fis = [FloatImage(a.ctypes.data_as(C.POINTER(C.c_float)), a.shape[1], a.shape[0]) for a in arrays]
    return fis, (C.POINTER(FloatImage) * len(fis))(*[C.pointer(x) for x in fis])


class Buffers:
    """Page-locked host buffers of one workload: frames, arm (b)'s float frames, edge maps of both arms, outputs."""

    def __init__(self, ctx, frames, jets, edges):
        import numpy as np
        from slowflow_b200 import ColorImage, Image
        from slowflow_b200.image import image_t
        h, w = frames[0].shape[:2]
        self.floats = [ColorImage(w, h) for _ in frames]
        self.out = {a: [[Image(w, h) for _ in range(jets)] for _ in range(5)] for a in "ab"}
        self.arrays = [(C.POINTER(image_t) * jets)(*[C.pointer(x.c) for x in ps]) for ps in self.out["a"]]
        self.edges_orig = edges
        self.edges_a = [np.empty_like(e) for e in edges]
        self.edges_b = [np.empty_like(edges[k + back]) for k in range(jets) for back in (0, 1)]  # one per window
        self.bufs = (list(frames) + [f.buf for f in self.floats] + [x.buf for a in "ab" for ps in self.out[a] for x in ps] + self.edges_a +
                     self.edges_b)
        sjb.register(ctx.lib, self.bufs)
        self.lib = ctx.lib

    def refresh_edges(self, jets):
        import numpy as np
        for d, s in zip(self.edges_a, self.edges_orig):
            np.copyto(d, s)
        for i, d in enumerate(self.edges_b):
            np.copyto(d, self.edges_orig[i // 2 + i % 2])

    def release(self):
        for b in self.bufs:
            self.lib.sfgpu_host_unregister(b.ctypes.data)


def arm_call(ctx, frames, p, ep, jets, fwd_m, back_m, bf):
    from slowflow_b200.api import EpicStats, FrameInt
    from slowflow_b200.params import MTParams
    q = MTParams.from_buffer_copy(bytes(p))
    h, w = frames[0].shape[:2]
    fa = (FrameInt * len(frames))(*[FrameInt(w, h, 3, f.strides[0], f.ctypes.data) for f in frames])
    fm, bm, ed = float_images(fwd_m), float_images(back_m), float_images(bf.edges_a)
    st = (EpicStats * (2 * jets))()
    t0 = time.perf_counter()
    rc = ctx.lib.sfgpu_slow_flow_jets_epic(ctx.h, len(frames), fa, 8, 1.0, 0, jets, C.byref(q), 0, None, fm[1], bm[1], ed[1], C.byref(ep),
                                           *bf.arrays, st)
    dt = time.perf_counter() - t0
    if rc != 0:
        raise RuntimeError("sfgpu_slow_flow_jets_epic: %s" % ctx.lib.sfgpu_last_error().decode())
    return dt, [tuple(getattr(s, f) for f, _ in EpicStats._fields_) for s in st]


def arm_composed(ctx, frames, p, ep, jets, fwd_m, back_m, bf):
    import numpy as np
    from slowflow_b200.api import EpicStats
    from slowflow_b200.params import MTParams
    q = MTParams.from_buffer_copy(bytes(p))
    steps = p.S - 1
    F = 2 * steps + 1
    o = bf.out["b"]
    inv, sc = np.float32(1) / np.float32(steps), np.float32(steps)
    stats = []
    t0 = time.perf_counter()
    for f, im in zip(frames, bf.floats):  # convertTo(CV_32F) + colorMat2colorImg into the page-locked planes
        im.array[:] = np.moveaxis(f, 2, 0)
    ctx.normalize(bf.floats, q)
    ctx.mt_frame_cache(2 * F)  # after normalize(), as the driver does
    try:
        for k0 in range(0, jets, CHUNK):
            ks = range(k0, min(jets, k0 + CHUNK))
            refs = {r: ctx.rgb_to_lab(bf.floats[r * steps + steps]) for r in range(k0, ks[-1] + 2)} if ep.saliency_th != 0 else None
            fx, fy, ims, ms, es = [], [], [], [], []
            for k in ks:
                for back in (0, 1):
                    fx.append(o[2 if back else 0][k])
                    fy.append(o[3 if back else 1][k])
                    ims.append(refs[k + back] if refs else bf.floats[(k + back) * steps + steps])
                    ms.append((back_m if back else fwd_m)[k])
                    es.append(bf.edges_b[2 * k + back])
            st = ctx.epic_batch(fx, fy, ims, ms, es, ep)
            stats += [tuple(getattr(s, f) for f, _ in EpicStats._fields_) for s in st]
            for x in fx + fy:
                np.multiply(x.buf, inv, out=x.buf)
            for k in ks:
                b = k * steps
                for back in (0, 1):
                    wx, wy = o[2 if back else 0][k], o[3 if back else 1][k]
                    if back:
                        ctx.variational_mt(wx, wy, [bf.floats[b + 3 * steps - i] for i in range(F)], q)
                    else:
                        ctx.variational_mt(wx, wy, bf.floats[b:b + F], q, None, o[4][k])
                    np.multiply(wx.buf, sc, out=wx.buf)
                    np.multiply(wy.buf, sc, out=wy.buf)
    finally:
        ctx.mt_frame_cache(0)
    return time.perf_counter() - t0, stats


def main():
    a = parse()
    os.makedirs(a.out, exist_ok=True)
    from slowflow_b200 import Context
    from slowflow_b200.api import epic_params_default
    res = {"device": sjb.device_info(), "host_buffers": "page-locked (sfgpu_host_register)", "workloads": []}
    print(res["device"])
    ctx = Context(0)
    ep = epic_params_default()
    for name in a.workloads.split(","):
        w, h, S, jets, kind, n_matches = WORKLOADS[name]
        steps = S - 1
        p = sjb.params(kind, S, 8)
        frames = sjb.make_frames(w, h, 1 + (jets + 2) * steps, 8, steps)
        fwd_m, back_m, edges = epic_inputs(w, h, steps, jets, n_matches)
        bf = Buffers(ctx, frames, jets, edges)
        try:
            ta, tb = [], []
            for rep in range(a.reps + 1):  # repetition 0 is the warm-up of both arms
                bf.refresh_edges(jets)
                t, sa = arm_call(ctx, frames, p, ep, jets, fwd_m, back_m, bf)
                t2, sb = arm_composed(ctx, frames, p, ep, jets, fwd_m, back_m, bf)
                if rep:
                    ta.append(t)
                    tb.append(t2)
                assert sa == sb, "EPIC stats differ"
                for k in range(5):
                    for x, y in zip(bf.out["a"][k], bf.out["b"][k]):
                        assert x.buf.tobytes() == y.buf.tobytes(), "arms differ (%s)" % ("fwd_x fwd_y back_x back_y occlusions".split()[k])
                for i, e in enumerate(bf.edges_b):
                    assert e.tobytes() == bf.edges_a[i // 2 + i % 2].tobytes(), "edge maps differ"
        finally:
            bf.release()
        s_a, s_b = sjb.summary(ta), sjb.summary(tb)
        rate = lambda s: {k: 1e3 * jets / s[v] for k, v in (("median", "median_ms"), ("min", "max_ms"), ("max", "min_ms"))}
        row = {"name": name, "width": w, "height": h, "S": S, "bits": 8, "jets": jets, "n_frames": len(frames), "params": kind,
               "matches_per_window": n_matches, "epic": {f: (getattr(ep, f).decode() if f == "method" else getattr(ep, f))
                                                         for f, _ in ep._fields_},
               "call": s_a, "composed": s_b, "jets_per_s_call": rate(s_a), "jets_per_s_composed": rate(s_b), "outputs_equal": True}
        res["workloads"].append(row)
        print("%s: call %.1f ms (%.2f jets/s, %.2f..%.2f), composed %.1f ms (%.2f jets/s, %.2f..%.2f), ratio %.2f; outputs equal" %
              (name, s_a["median_ms"], row["jets_per_s_call"]["median"], row["jets_per_s_call"]["min"], row["jets_per_s_call"]["max"],
               s_b["median_ms"], row["jets_per_s_composed"]["median"], row["jets_per_s_composed"]["min"],
               row["jets_per_s_composed"]["max"], s_b["median_ms"] / s_a["median_ms"]))
        sys.stdout.flush()
    ctx.close()
    with open(os.path.join(a.out, "slow_flow_jets_epic_bench.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
