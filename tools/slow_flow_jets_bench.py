#!/usr/bin/env python3
"""The Slow Flow jet loop over one integer sequence: one sfgpu_slow_flow_jets call against the composition it replaces.

Arms, run alternately in one process after one warm-up call of each per workload, with page-locked host buffers:
  (a) ctx.slow_flow_jets: integer frames cross PCIe (twice: statistics pass, then the jets), everything else on the device;
  (b) the composition through the Python API, as tools/slow_flow_gpu.cpp runs it: integer -> float32 frames on the host,
      ctx.normalize over the whole sequence, then per window ctx.variational_mt with the frame cache on
      (sfgpu_mt_frame_cache) and the flow multiplied by S-1 on the host.  Its float frames and flow planes are page-locked
      once, outside the timed region, like the driver does before its loop.
Every call ends with a stream synchronise, so a host clock around it measures the device work plus what the host adds.
The outputs of both arms (forward / backward flows and occlusion labels) are compared bit for bit on every repetition.

Also reported: arm (a)'s statistics pass on its own (sfgpu_get_mt_stats setup_ms), and the device-busy share of arm (a):
the union of its kernels' execution intervals (torch.profiler, CUDA activities, one extra profiled call) over that call's
wall time.  The card's name, power limit and top SM clock are read in the same run.

    python tools/slow_flow_jets_bench.py --out DIR [--reps 5] [--workloads NAME,...]
Writes DIR/slow_flow_jets_bench.json and prints a summary.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# name: (width, height, S, bits, jets, parameter set).  "driver": tools/driver_bench.py (Geman-McClure eps 0.5, occlusion
# reasoning, 2 alternations); "config4": BASELINE config 4 (the same with 3 pyramid layers).  Every frame of these
# sequences is 1.3 / 2.6 / 3.7 MB of integers and the windows' working set is far beyond the 126 MB L2.
WORKLOADS = {
    "1280x1024_u8": (1280, 1024, 3, 8, 16, "driver"),
    "1280x1024_u16": (1280, 1024, 3, 16, 16, "driver"),
    "2560x1440_config4_u8": (2560, 1440, 3, 8, 4, "config4"),
}


def parse():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="directory for slow_flow_jets_bench.json")
    ap.add_argument("--reps", type=int, default=5, help="timed repetitions per arm and workload")
    ap.add_argument("--workloads", default=",".join(WORKLOADS), help="comma-separated subset of " + ", ".join(WORKLOADS))
    return ap.parse_args()


def device_info():
    """The card's name, power limit and top SM clock (read-only query)."""
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True,
                           timeout=60)
        return r.stdout.strip()
    except Exception as e:  # the numbers are not worth much without it, but the run can go on
        return "nvidia-smi failed: %r" % (e,)


def params(kind, S, bits):
    from slowflow_b200 import mt_params_default
    p = mt_params_default()
    p.S, p.hbit = S, 1 if bits == 16 else 0
    p.niter_alter = 2
    p.robust_color, p.robust_color_eps = 4, 0.5
    p.occlusion_reasoning = 1
    p.layers = 3 if kind == "config4" else 1
    return p


_TEXTURE = {}


def make_frames(w, h, n, bits, steps):
    """The sequence of tools/driver_bench.py (frame k = synth.frame(w, h, k - steps)) in (H, W, 3) cv::Mat layout; 16-bit
    frames hold the same images scaled to 12 bits."""
    import numpy as np
    from slowflow_b200 import synth
    key = (w, h, n, steps)
    if key not in _TEXTURE:
        _TEXTURE.clear()
        _TEXTURE[key] = [np.moveaxis(synth.frame(w, h, k - steps), 0, 2) for k in range(n)]
    top = 255.0 if bits == 8 else 4095.0
    dt = np.uint8 if bits == 8 else np.uint16
    return [np.ascontiguousarray(np.rint(f * (top / 255.0)).clip(0, top).astype(dt)) for f in _TEXTURE[key]]


def register(lib, bufs):
    for b in bufs:
        if lib.sfgpu_host_register(b.ctypes.data, b.nbytes) != 0:
            raise RuntimeError("sfgpu_host_register failed: %s" % lib.sfgpu_last_error().decode())


class Buffers:
    """The page-locked host buffers of one workload: frames, arm (b)'s float frames, both arms' outputs."""

    def __init__(self, ctx, frames, S, jets):
        import ctypes as C
        from slowflow_b200 import ColorImage, Image
        from slowflow_b200.image import image_t
        h, w = frames[0].shape[:2]
        self.floats = [ColorImage(w, h) for _ in frames]
        self.out = {a: [[Image(w, h) for _ in range(jets)] for _ in range(5)] for a in "ab"}
        IP = C.POINTER(image_t)
        self.arrays = [(IP * jets)(*[C.pointer(x.c) for x in ps]) for ps in self.out["a"]]
        self.bufs = list(frames) + [f.buf for f in self.floats] + [x.buf for a in "ab" for ps in self.out[a] for x in ps]
        register(ctx.lib, self.bufs)
        self.lib = ctx.lib

    def release(self):
        for b in self.bufs:
            self.lib.sfgpu_host_unregister(b.ctypes.data)


def arm_jets(ctx, frames, p, jets, bf):
    import ctypes as C
    from slowflow_b200.api import FrameInt
    from slowflow_b200.params import MTParams
    q = MTParams.from_buffer_copy(bytes(p))
    h, w = frames[0].shape[:2]
    fa = (FrameInt * len(frames))(*[FrameInt(w, h, 3, f.strides[0], f.ctypes.data) for f in frames])
    bits = frames[0].dtype.itemsize * 8
    t0 = time.perf_counter()
    rc = ctx.lib.sfgpu_slow_flow_jets(ctx.h, len(frames), fa, bits, 1.0, 0, jets, C.byref(q), 0, None, *bf.arrays)
    dt = time.perf_counter() - t0
    if rc != 0:
        raise RuntimeError("sfgpu_slow_flow_jets: %s" % ctx.lib.sfgpu_last_error().decode())
    return dt, ctx.mt_stats().setup_ms * 1e-3


def arm_composed(ctx, frames, p, jets, bf):
    import numpy as np
    from slowflow_b200.params import MTParams
    q = MTParams.from_buffer_copy(bytes(p))
    steps = p.S - 1
    F = 2 * steps + 1
    o = bf.out["b"]
    t0 = time.perf_counter()
    for f, im in zip(frames, bf.floats):  # convertTo(CV_32F) + colorMat2colorImg into the page-locked planes
        im.array[:] = np.moveaxis(f, 2, 0)
    ctx.normalize(bf.floats, q)
    ctx.mt_frame_cache(2 * F)  # after normalize(), as the driver does
    try:
        for j in range(jets):
            b = j * steps
            for back in (False, True):
                wx, wy = o[2 if back else 0][j], o[3 if back else 1][j]
                wx.buf[:] = 0
                wy.buf[:] = 0
                win = [bf.floats[b + 3 * steps - i] for i in range(F)] if back else bf.floats[b:b + F]
                if back:
                    ctx.variational_mt(wx, wy, win, q)
                else:
                    ctx.variational_mt(wx, wy, win, q, None, o[4][j])
                np.multiply(wx.buf, np.float32(steps), out=wx.buf)
                np.multiply(wy.buf, np.float32(steps), out=wy.buf)
    finally:
        ctx.mt_frame_cache(0)
    return time.perf_counter() - t0


def busy_share(ctx, frames, p, jets, bf):
    """Union of the kernel intervals of one arm (a) call over its wall time (torch.profiler, CUDA activities)."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
    except Exception as e:
        return "not measured (%r)" % (e,)
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        wall, _ = arm_jets(ctx, frames, p, jets, bf)
    iv = sorted((e.time_range.start, e.time_range.end) for e in prof.events()
                if getattr(e, "device_type", None) is not None and "cuda" in str(e.device_type).lower() and "memcpy" not in e.name.lower()
                and "memset" not in e.name.lower())
    if not iv:
        return "not measured (no kernel events)"
    busy, cur_s, cur_e = 0.0, iv[0][0], iv[0][1]
    for s, e in iv[1:]:
        if s > cur_e:
            busy += cur_e - cur_s
            cur_s, cur_e = s, e
        else:
            cur_e = max(cur_e, e)
    busy += cur_e - cur_s
    return {"kernel_busy_ms": busy * 1e-3, "wall_ms_profiled": wall * 1e3, "share": busy * 1e-6 / wall, "kernels": len(iv)}


def summary(ts):
    ts = sorted(ts)
    return {"median_ms": 1e3 * ts[len(ts) // 2], "min_ms": 1e3 * ts[0], "max_ms": 1e3 * ts[-1], "reps": len(ts)}


def main():
    a = parse()
    os.makedirs(a.out, exist_ok=True)
    from slowflow_b200 import Context
    res = {"device": device_info(), "host_buffers": "page-locked (sfgpu_host_register)", "workloads": []}
    print(res["device"])
    ctx = Context(0)
    for name in a.workloads.split(","):
        w, h, S, bits, jets, kind = WORKLOADS[name]
        steps = S - 1
        p = params(kind, S, bits)
        frames = make_frames(w, h, 1 + (jets + 2) * steps, bits, steps)
        bf = Buffers(ctx, frames, S, jets)
        try:
            arm_jets(ctx, frames, p, jets, bf)  # warm-up: workspaces, io area, module loads
            arm_composed(ctx, frames, p, jets, bf)
            ta, tb, t1 = [], [], []
            for _ in range(a.reps):
                t, s1 = arm_jets(ctx, frames, p, jets, bf)
                ta.append(t)
                t1.append(s1)
                tb.append(arm_composed(ctx, frames, p, jets, bf))
                for k in range(5):
                    for x, y in zip(bf.out["a"][k], bf.out["b"][k]):
                        assert x.buf.tobytes() == y.buf.tobytes(), "arms differ (%s)" % ("fwd_x fwd_y back_x back_y occlusions".split()[k])
            busy = busy_share(ctx, frames, p, jets, bf)
        finally:
            bf.release()
        sa, sb = summary(ta), summary(tb)
        row = {"name": name, "width": w, "height": h, "S": S, "bits": bits, "jets": jets, "n_frames": len(frames), "params": kind,
               "jets_call": sa, "composed": sb, "jets_per_s_call": {k: 1e3 * jets / sa[v] for k, v in
                                                                    (("median", "median_ms"), ("min", "max_ms"), ("max", "min_ms"))},
               "jets_per_s_composed": {k: 1e3 * jets / sb[v] for k, v in (("median", "median_ms"), ("min", "max_ms"), ("max", "min_ms"))},
               "statistics_pass": summary(t1), "device_busy_call": busy, "outputs_equal": True}
        res["workloads"].append(row)
        print("%s: call %.1f ms (%.1f jets/s, %.1f..%.1f), composed %.1f ms (%.1f jets/s, %.1f..%.1f), statistics pass %.1f ms, "
              "busy %s; outputs equal" % (name, sa["median_ms"], row["jets_per_s_call"]["median"], row["jets_per_s_call"]["min"],
                                          row["jets_per_s_call"]["max"], sb["median_ms"], row["jets_per_s_composed"]["median"],
                                          row["jets_per_s_composed"]["min"], row["jets_per_s_composed"]["max"],
                                          row["statistics_pass"]["median_ms"], busy if isinstance(busy, str) else "%.3f" % busy["share"]))
        sys.stdout.flush()
    ctx.close()
    with open(os.path.join(a.out, "slow_flow_jets_bench.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
