#!/usr/bin/env python3
"""Throughput of EPIC on many images of one geometry: N sequential sfgpu_epic calls against one sfgpu_epic_batch of N.

Arms, run alternately in one process after a warm-up of every shape:
  (a) N sequential ctx.epic calls on one context;
  (b) one ctx.epic_batch of the N items;
  (c) N host threads, each with its own context, calling epic at the same time (reported only: what a multi-threaded
      caller gets without the batch entry).
Each call ends with a stream synchronise, so a host clock around the calls measures the device work.  The outputs of (b)
and (c) are compared bit for bit with (a) on every timed repetition.  With --parent-lib the N = 1 single call and batch of
one are also timed against sfgpu_epic of another build of the library, alternating in the same process.  The phase split
of one batched call (SLOWFLOW_GPU_TRACE=1, stderr of the library) is recorded per geometry for N = 1 and the largest N.

The 1024x436 working set (a few tens of MB per item) fits the B200's 126 MB L2; 2560x1440 does not.

    python tools/epic_batch_bench.py --out DIR [--reps 7] [--ns 1,2,4,8] [--parent-lib PATH]
Writes DIR/epic_batch_bench.json and prints a summary.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GEOMETRIES = [(1024, 436, 5000), (2560, 1440, 20000)]  # the EpicFlow paper's Sintel size; the README's 2560x1440 case


def parse():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="directory for epic_batch_bench.json")
    ap.add_argument("--reps", type=int, default=7, help="timed repetitions per arm and shape (>= 5)")
    ap.add_argument("--ns", default="1,2,4,8", help="batch sizes")
    ap.add_argument("--geometries", default=",".join("%dx%d:%d" % g for g in GEOMETRIES), help="WxH:matches,...")
    ap.add_argument("--parent-lib", default=None, help="another build of libslowflow_gpu.so for the N = 1 comparison")
    return ap.parse_args()


def device_info():
    """The card's name, power limit and top SM clock (read-only query)."""
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True,
                           timeout=60)
        return r.stdout.strip()
    except Exception as e:  # the numbers are not worth much without it, but the run can go on
        return "nvidia-smi failed: %r" % (e,)


def make_items(w, h, n_matches, count):
    from slowflow_b200 import ColorImage, synth
    out = []
    for k in range(count):
        im, m, edges = synth.epic_case(w, h, n_matches, seed=7000 + 13 * k)
        out.append((ColorImage.from_array(im), m, edges))
    return out


def planes(w, h, n):
    from slowflow_b200 import Image
    return [(Image(w, h), Image(w, h)) for _ in range(n)]


def outputs(fl):
    return [(fx.buf.tobytes(), fy.buf.tobytes()) for fx, fy in fl]


def arm_sequential(ctx, items, w, h):
    fl, es = planes(w, h, len(items)), [e.copy() for _, _, e in items]
    t0 = time.perf_counter()
    for (im, m, _), (fx, fy), e in zip(items, fl, es):
        ctx.epic(fx, fy, im, m, e, None)
    return time.perf_counter() - t0, outputs(fl)


def arm_batch(ctx, items, w, h):
    fl, es = planes(w, h, len(items)), [e.copy() for _, _, e in items]
    t0 = time.perf_counter()
    ctx.epic_batch([f[0] for f in fl], [f[1] for f in fl], [i[0] for i in items], [i[1] for i in items], es, None)
    return time.perf_counter() - t0, outputs(fl)


def arm_threads(ctxs, items, w, h):
    n = len(items)
    fl, es = planes(w, h, n), [e.copy() for _, _, e in items]
    go, err = threading.Barrier(n + 1), []

    def work(k):
        go.wait()
        try:
            im, m, _ = items[k]
            ctxs[k].epic(fl[k][0], fl[k][1], im, m, es[k], None)
        except Exception as e:  # pragma: no cover
            err.append(repr(e))

    th = [threading.Thread(target=work, args=(k,)) for k in range(n)]
    for t in th:
        t.start()
    go.wait()
    t0 = time.perf_counter()
    for t in th:
        t.join()
    dt = time.perf_counter() - t0
    if err:
        raise RuntimeError(err[0])
    return dt, outputs(fl)


def stats_of(times, n):
    ips = sorted(n / t for t in times)
    return {"images_per_s_median": ips[len(ips) // 2], "images_per_s_min": ips[0], "images_per_s_max": ips[-1],
            "spread_pct": 100.0 * (ips[-1] - ips[0]) / ips[len(ips) // 2], "call_ms": [1e3 * t for t in times]}


def traced(fn):
    """Runs fn with SLOWFLOW_GPU_TRACE=1 and returns what the library wrote to stderr."""
    os.environ["SLOWFLOW_GPU_TRACE"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile() as f:
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["SLOWFLOW_GPU_TRACE"]
        f.seek(0)
        return f.read().decode(errors="replace")


def context_on(path):
    """A Context whose calls go to the library at `path` (another build, loaded next to this one; only epic is used)."""
    from slowflow_b200 import Context
    from slowflow_b200.api import _check, load_library
    lib = C.CDLL(path, mode=os.RTLD_LOCAL | os.RTLD_NOW)
    lib.sfgpu_last_error.restype = C.c_char_p
    lib.sfgpu_create.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
    lib.sfgpu_destroy.argtypes = [C.c_void_p]
    lib.sfgpu_destroy.restype = None
    lib.sfgpu_epic.argtypes = load_library().sfgpu_epic.argtypes
    c = Context.__new__(Context)
    c.lib, c.device, h = lib, 0, C.c_void_p()
    _check(lib, lib.sfgpu_create(0, None, C.byref(h)), "sfgpu_create")
    c.h = h
    return c


def main():
    a = parse()
    if a.reps < 5:
        sys.exit("--reps must be >= 5")
    ns = [int(x) for x in a.ns.split(",")]
    geos = []
    for g in a.geometries.split(","):
        wh, m = g.split(":")
        w, h = wh.split("x")
        geos.append((int(w), int(h), int(m)))
    os.makedirs(a.out, exist_ok=True)

    from slowflow_b200 import Context
    from slowflow_b200.api import library_path
    result = {"device": device_info(), "library": os.path.relpath(library_path(), ROOT), "reps": a.reps, "ns": ns, "geometries": [], "parent": None}
    ctx = Context(0)
    ctxs = [Context(0) for _ in range(max(ns))]
    items = {g: make_items(g[0], g[1], g[2], max(ns)) for g in geos}

    # warm-up of every shape and arm
    for g in geos:
        for n in ns:
            arm_sequential(ctx, items[g][:n], g[0], g[1])
            arm_batch(ctx, items[g][:n], g[0], g[1])
            arm_threads(ctxs[:n], items[g][:n], g[0], g[1])

    times = {(g, n, arm): [] for g in geos for n in ns for arm in "abc"}
    equal = {(g, n, arm): True for g in geos for n in ns for arm in "bc"}
    for _ in range(a.reps):
        for g in geos:
            for n in ns:
                w, h = g[0], g[1]
                ta, oa = arm_sequential(ctx, items[g][:n], w, h)
                tb, ob = arm_batch(ctx, items[g][:n], w, h)
                tc, oc = arm_threads(ctxs[:n], items[g][:n], w, h)
                times[(g, n, "a")].append(ta)
                times[(g, n, "b")].append(tb)
                times[(g, n, "c")].append(tc)
                equal[(g, n, "b")] &= ob == oa
                equal[(g, n, "c")] &= oc == oa

    for g in geos:
        w, h, m = g
        entry = {"width": w, "height": h, "matches": m, "by_n": []}
        for n in ns:
            e = {"n": n, "batch_bit_identical_to_sequential": equal[(g, n, "b")], "threads_bit_identical_to_sequential": equal[(g, n, "c")]}
            for arm, name in (("a", "sequential"), ("b", "batch"), ("c", "threads")):
                e[name] = stats_of(times[(g, n, arm)], n)
            e["batch_over_sequential"] = e["batch"]["images_per_s_median"] / e["sequential"]["images_per_s_median"]
            entry["by_n"].append(e)
        entry["trace"] = {}
        for n in sorted({1, max(ns)}):
            entry["trace"]["batch_n%d" % n] = traced(lambda: arm_batch(ctx, items[g][:n], w, h))
        result["geometries"].append(entry)

    if a.parent_lib:
        parent = context_on(os.path.abspath(a.parent_lib))
        par = {"library": a.parent_lib, "by_geometry": []}
        for g in geos:
            w, h = g[0], g[1]
            one = items[g][:1]
            arm_sequential(parent, one, w, h)
            t = {"parent_epic": [], "epic": [], "epic_batch_n1": []}
            same = True
            for _ in range(4 * a.reps):
                tp, op = arm_sequential(parent, one, w, h)
                ts, os_ = arm_sequential(ctx, one, w, h)
                tb, ob = arm_batch(ctx, one, w, h)
                t["parent_epic"].append(tp)
                t["epic"].append(ts)
                t["epic_batch_n1"].append(tb)
                same &= op == os_ == ob
            par["by_geometry"].append({"width": w, "height": h, "bit_identical_to_parent": same, **{k: stats_of(v, 1) for k, v in t.items()}})
        parent.close()
        result["parent"] = par

    path = os.path.join(a.out, "epic_batch_bench.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(result["device"])
    for entry in result["geometries"]:
        for e in entry["by_n"]:
            print("%dx%d N=%d  images/s: sequential %.1f  batch %.1f (x%.2f)  threads %.1f   spread %% a/b/c %.1f/%.1f/%.1f  identical b=%s c=%s" % (
                entry["width"], entry["height"], e["n"], e["sequential"]["images_per_s_median"], e["batch"]["images_per_s_median"],
                e["batch_over_sequential"], e["threads"]["images_per_s_median"], e["sequential"]["spread_pct"], e["batch"]["spread_pct"],
                e["threads"]["spread_pct"], e["batch_bit_identical_to_sequential"], e["threads_bit_identical_to_sequential"]))
    if result["parent"]:
        for p in result["parent"]["by_geometry"]:
            print("%dx%d N=1 ms (median of %d): parent epic %.3f  epic %.3f  batch of one %.3f  identical=%s" % (
                p["width"], p["height"], len(p["epic"]["call_ms"]), 1e3 / p["parent_epic"]["images_per_s_median"],
                1e3 / p["epic"]["images_per_s_median"], 1e3 / p["epic_batch_n1"]["images_per_s_median"], p["bit_identical_to_parent"]))
    print("wrote", path)


if __name__ == "__main__":
    main()
