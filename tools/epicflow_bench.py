#!/usr/bin/env python3
"""The EpicFlow two-step over consecutive pairs: one sfgpu_epicflow_sequence call against the GPU-only composition.

Arms, run alternately in one process after one warm-up call of each per shape, with page-locked host buffers:
  (a) ctx.epicflow_sequence: Lab on the device, the interpolated flows stay resident, each frame crosses PCIe once;
  (b) ctx.rgb_to_lab per frame, then ctx.epic_batch in batches of 8 pairs, then ctx.variational_sequence.
(b) converts to Lab on the GPU too, so (a) - (b) is the gain of the transfers and overlap saved, not of the host conversion.
Every call ends with a stream synchronise, so a host clock around the calls measures the device work.  The flows of both
arms are compared bit for bit on every timed repetition.  Where the reference build (oracle/_ref/libsf_ref.so) exports
rgb_to_lab, its host time per frame is reported too; otherwise it is "not measured".

At 2560x1440 a chunk's working set is several GB, far beyond the B200's 126 MB L2; at 1024x436 a pair's inputs fit it.

    python tools/epicflow_bench.py --out DIR [--reps 5] [--pairs 8,24] [--geometries 1024x436:5000,2560x1440:20000]
Writes DIR/epicflow_bench.json and prints a summary.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GEOMETRIES = [(1024, 436, 5000), (2560, 1440, 20000)]
BATCH = 8  # pairs per epic_batch call in arm (b): the chunk size of sfgpu_epicflow_sequence


def parse():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="directory for epicflow_bench.json")
    ap.add_argument("--reps", type=int, default=5, help="timed repetitions per arm and shape")
    ap.add_argument("--pairs", default="8,24", help="numbers of pairs")
    ap.add_argument("--geometries", default=",".join("%dx%d:%d" % g for g in GEOMETRIES), help="WxH:matches,...")
    return ap.parse_args()


def device_info():
    """The card's name, power limit and top SM clock (read-only query)."""
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True,
                           timeout=60)
        return r.stdout.strip()
    except Exception as e:  # the numbers are not worth much without it, but the run can go on
        return "nvidia-smi failed: %r" % (e,)


def make_inputs(w, h, n_matches, n):
    """n + 1 frames, and per pair seeded matches and edge costs (one synthetic case, shifted and perturbed per pair)."""
    import numpy as np
    from slowflow_b200 import ColorImage, synth
    _, m0, e0 = synth.epic_case(w, h, n_matches, seed=9100)
    base = synth.frame(w, h, 0)
    frames, ms, es = [], [], []
    for t in range(n + 1):  # the texture moved by t pixels: cheap to make at 2560x1440, distinct per frame
        frames.append(ColorImage.from_array(np.roll(base, t, axis=2)))
    for k in range(n):
        r = np.random.RandomState(9200 + k)
        m = m0.copy()
        m[:, 2:] += r.uniform(-0.5, 0.5, (m.shape[0], 2)).astype(np.float32)
        ms.append(m)
        es.append(np.clip(e0 + 0.05 * r.rand(h, w), 0.0, 1.0).astype(np.float32))
    return frames, ms, es


def register(lib, bufs):
    for b in bufs:
        if lib.sfgpu_host_register(b.ctypes.data, b.nbytes) != 0:
            raise RuntimeError("sfgpu_host_register failed: %s" % lib.sfgpu_last_error().decode())


class Buffers:
    """The page-locked host buffers of one shape: flows and edge copies per arm, Lab images for arm (b)."""

    def __init__(self, lib, frames, es):
        from slowflow_b200 import ColorImage, Image
        w, h, n = frames[0].width, frames[0].height, len(es)
        self.fl = {a: [(Image(w, h), Image(w, h)) for _ in range(n)] for a in "ab"}
        self.edges = {a: [e.copy() for e in es] for a in "ab"}
        self.labs = [ColorImage(w, h) for _ in range(n)]
        self.bufs = [f.buf for f in frames] + [lab.buf for lab in self.labs] + list(self.edges["a"]) + list(self.edges["b"])
        self.bufs += [p.buf for a in "ab" for f in self.fl[a] for p in f]
        register(lib, self.bufs)
        self.lib = lib

    def release(self):
        for b in self.bufs:
            self.lib.sfgpu_host_unregister(b.ctypes.data)


def arm_sequence(ctx, frames, ms, es, bf):
    for e, src in zip(bf.edges["a"], es):
        e[:] = src
    fl = bf.fl["a"]
    t0 = time.perf_counter()
    ctx.epicflow_sequence(frames, ms, bf.edges["a"], [f[0] for f in fl], [f[1] for f in fl])
    return time.perf_counter() - t0


def arm_composed(ctx, frames, ms, es, bf):
    n = len(ms)
    for e, src in zip(bf.edges["b"], es):
        e[:] = src
    fl = bf.fl["b"]
    t0 = time.perf_counter()
    for k in range(n):  # into the page-locked Lab images (ctx.rgb_to_lab would return a new pageable one)
        if ctx.lib.sfgpu_rgb_to_lab(ctx.h, bf.labs[k].ptr(), frames[k].ptr()) != 0:
            raise RuntimeError("sfgpu_rgb_to_lab: %s" % ctx.lib.sfgpu_last_error().decode())
    for k0 in range(0, n, BATCH):
        sl = slice(k0, min(n, k0 + BATCH))
        ctx.epic_batch([f[0] for f in fl[sl]], [f[1] for f in fl[sl]], bf.labs[sl], ms[sl], bf.edges["b"][sl])
    ctx.variational_sequence(frames, [f[0] for f in fl], [f[1] for f in fl])
    return time.perf_counter() - t0


def host_lab_ms(frame, reps=3):
    """Host time of the reference's rgb_to_lab on one frame (ms), or None without the reference build."""
    from oracle.pyoracle import have_reference, REF_SO
    from slowflow_b200.image import color_image_t
    if not have_reference():
        return None
    lib = C.CDLL(REF_SO, mode=os.RTLD_LOCAL)
    if not hasattr(lib, "rgb_to_lab"):
        return None
    lib.rgb_to_lab.argtypes = [C.POINTER(color_image_t)]
    lib.rgb_to_lab.restype = C.POINTER(color_image_t)
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = lib.rgb_to_lab(frame.ptr())
        dt = (time.perf_counter() - t0) * 1e3
        best = dt if best is None else min(best, dt)
        if hasattr(lib, "color_image_delete"):
            lib.color_image_delete.argtypes = [C.POINTER(color_image_t)]
            lib.color_image_delete(out)
    return best


def summary(ts):
    ts = sorted(ts)
    return {"median_ms": 1e3 * ts[len(ts) // 2], "min_ms": 1e3 * ts[0], "max_ms": 1e3 * ts[-1], "reps": len(ts)}


def main():
    a = parse()
    os.makedirs(a.out, exist_ok=True)
    from slowflow_b200 import Context
    geos = [tuple(int(x) for x in g.replace(":", "x").split("x")) for g in a.geometries.split(",")]
    pairs = [int(x) for x in a.pairs.split(",")]
    res = {"device": device_info(), "host_buffers": "page-locked (sfgpu_host_register)", "epic_batch_size_arm_b": BATCH, "shapes": []}
    print(res["device"])
    ctx = Context(0)
    for (w, h, nm) in geos:
        for n in pairs:
            frames, ms, es = make_inputs(w, h, nm, n)
            bf = Buffers(ctx.lib, frames, es)
            try:
                arm_sequence(ctx, frames, ms, es, bf)  # warm-up of the shape: workspaces, arenas, module loads
                arm_composed(ctx, frames, ms, es, bf)
                ta, tb = [], []
                for _ in range(a.reps):
                    ta.append(arm_sequence(ctx, frames, ms, es, bf))
                    tb.append(arm_composed(ctx, frames, ms, es, bf))
                    for (ax, ay), (bx, by) in zip(bf.fl["a"], bf.fl["b"]):
                        assert ax.buf.tobytes() == bx.buf.tobytes() and ay.buf.tobytes() == by.buf.tobytes(), "arms differ"
                    assert all(x.tobytes() == y.tobytes() for x, y in zip(bf.edges["a"], bf.edges["b"])), "edges differ"
            finally:
                bf.release()
            lab_ms = host_lab_ms(frames[0])
            sa, sb = summary(ta), summary(tb)
            row = {"width": w, "height": h, "matches": nm, "pairs": n, "sequence": sa, "composed": sb,
                   "speedup_median": sb["median_ms"] / sa["median_ms"], "flows_equal": True,
                   "host_rgb_to_lab_ms_per_frame": lab_ms if lab_ms is not None else "not measured"}
            res["shapes"].append(row)
            print("%dx%d %d matches, %2d pairs: sequence %8.1f ms (%.2f ms/pair), composed %8.1f ms (%.2f ms/pair), x%.3f; "
                  "flows equal; host rgb_to_lab %s" % (w, h, nm, n, sa["median_ms"], sa["median_ms"] / n, sb["median_ms"], sb["median_ms"] / n,
                                                       row["speedup_median"], "%.1f ms/frame" % lab_ms if lab_ms is not None else "not measured"))
            sys.stdout.flush()
    ctx.close()
    with open(os.path.join(a.out, "epicflow_bench.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
