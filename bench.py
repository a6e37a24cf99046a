#!/usr/bin/env python
"""bench.py -- refined flow fields / second at 2560x1440 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W                (our arm; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K --warmup W   (the reference's CPU path)
    python bench.py ... --dump-outputs DIR                        (also writes the last timed step's flows, see dump_outputs)

A "step" is one pass of the hot path over one batch: every rank refines `--pairs` consecutive
synthetic frame pairs at 2560x1440 with the reference's default two-frame parameters (5 outer x 1 inner
x 30 SOR sweeps, variational.c:85-98) -- BASELINE config 2, sharded as in config 5 (independent pairs,
no data-path collective, weak scaling).

  value     whole-job fields/s with inputs already resident in HBM (sfgpu_variational_dev)
  e2e       the same metric through the host-buffer C ABI: 8-bit frames as adaptiveFR.cpp:450-464 holds them
            (sfgpu_variational_sequence_u8) and fp32 flows in pinned host memory are copied H2D and the refined
            flows D2H inside the timed region; e2e.f32_frames = the same with fp32 frames
            (sfgpu_variational_sequence), e2e.legacy = the unmodified variational() entry on malloc'ed buffers
  roofline  SOR kernel: algorithmic bytes (44 B/px/sweep, SURVEY 8d) / CUDA-event time of the SOR launches
  cpu_baseline  the reference's CPU objects timed on this box's host cores (rank 0, N=1 only)
  secondary the multi-frame path (BASELINE configs 3 and 4): ms per window, executed iteration counts, host /
            kernel split, fraction of the fused streaming model, the reference's CPU seconds per outer iteration;
            EPIC interpolation; config 5's multi-frame secondary through the sharded window driver (slow_flow_gpu)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W_FULL, H_FULL = 2560, 1440
WORKLOAD = "two-frame variational refinement %dx%d, whole fields, 5 outer x 1 inner x 30 SOR sweeps (BASELINE config 2)"
SOR_BYTES_PER_PX_SWEEP = 44.0  # read a11' a12' a22' b1 b2 psi_h psi_v du dv (36) + write du dv (8)
DATA_BYTES_PER_PX = 52.0       # fused warp+derivatives+data term+laplacian model (SURVEY 8d)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=24,
                    help="frame pairs per rank and step (default 24: 10 steps = the 240 pairs of config 5)")
    ap.add_argument("--total-pairs", type=int, default=0,
                    help="strong-scaling variant (config 5 as one job): this many consecutive pairs of ONE sequence per step, "
                         "split over the ranks in contiguous ranges (slowflow_b200.shard.shard_range); overrides --pairs")
    ap.add_argument("--width", type=int, default=W_FULL)
    ap.add_argument("--height", type=int, default=H_FULL)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the multi-frame (config 3 / 4) secondary measurement")
    ap.add_argument("--sor-fuse", type=int, default=0)
    ap.add_argument("--sor-variant", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="GPU arm only: write the refined flows of the last timed step (rank 0) as DIR/flow_x.npy and "
                         "DIR/flow_y.npy, see dump_outputs")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs: the reference arm keeps no flows (it times the CPU path on a sample)")
    return a


# ----------------------------------------------------------------------------------------- helpers
def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class _StdoutToStderr:
    """The reference's CPU driver prints progress with cout ("layer 2:" ...); bench.py's stdout carries ONE JSON line, so the
    C-level stdout is pointed at stderr while reference code runs."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *a):
        try:
            import ctypes
            ctypes.CDLL(None).fflush(None)
        except Exception:
            pass
        os.dup2(self.saved, 1)
        os.close(self.saved)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


class CpuOracleRunner:
    """Times the CPU path on a bounded sample: `workers` processes (persistent pool, inputs generated
    before the clock starts), each refining one full-width strip of `strip_rows` rows per step with the
    two-frame defaults.  value = fields / wall time."""

    def __init__(self, width, height, strip_rows, workers):
        from oracle.pyoracle import have_reference
        self.width, self.height, self.rows, self.workers = width, height, strip_rows, workers
        self.kind = "reference" if have_reference() else "port"
        if self.kind == "reference":
            from oracle.pyoracle import Reference
            Reference()  # dlopen in the parent as well: the forked workers inherit the mapping
        self.pool = None
        if workers > 1:
            import multiprocessing as mp
            self.pool = mp.get_context("fork").Pool(workers)
            self.pool.map(_cpu_prepare, [(width, strip_rows)] * workers)
        else:
            _cpu_prepare((width, strip_rows))
        self.sample = "%d x (%dx%d = %.3f field) per step, two-frame defaults 5x1x30, %s, %d process(es)" % (
            workers, width, strip_rows, strip_rows / float(height),
            "reference objects oracle/_ref (-O3 -msse4)" if self.kind == "reference" else "oracle port", workers)

    def step(self):
        """-> (fields processed, seconds)"""
        jobs = [(self.width, self.rows, self.kind, k) for k in range(self.workers)]
        t0 = time.perf_counter()
        if self.pool:
            self.pool.map(_cpu_worker, jobs, chunksize=1)
        else:
            _cpu_worker(jobs[0])
        dt = time.perf_counter() - t0
        return self.workers * (self.width * self.rows) / float(self.width * self.height), dt

    def close(self):
        if self.pool:
            self.pool.close()
            self.pool.join()


_CPU_CACHE = {}


def _cpu_prepare(key):
    from slowflow_b200 import ColorImage, synth
    if key not in _CPU_CACHE:
        width, rows = key
        im1, im2, wx, wy = synth.two_frame_case(width, rows)
        _CPU_CACHE[key] = (ColorImage.from_array(im1), ColorImage.from_array(im2), wx, wy)
    return True


def _cpu_worker(job):
    width, rows, kind, k = job
    from slowflow_b200 import Image
    from oracle.pyoracle import Oracle, Reference
    _cpu_prepare((width, rows))
    a, b, wx, wy = _CPU_CACHE[(width, rows)]
    impl = Reference() if kind == "reference" else Oracle()
    x, y = Image.from_array(wx), Image.from_array(wy)
    impl.variational(x, y, a, b, None, 0)  # the reference's own lexicographic solver
    return float(x.array[0, 0])


def _bind_to_gpu_numa_node(index):
    """One host thread per device (north star): pin this process to the CPUs NVML reports as local to the GPU, so
    that its pinned staging buffers are allocated on the GPU's own NUMA node and H2D/D2H copies do not cross the
    socket interconnect (matters at 8 GPUs: ~25 GB/s up + 10 GB/s down per GPU).  Best effort; returns a note."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = (ncpu + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w in range(words) for b in range(64) if (mask[w] >> b) & 1 and 64 * w + b < ncpu]
        allowed = set(os.sched_getaffinity(0))
        cpus = [c for c in cpus if c in allowed]
        if cpus and len(cpus) < len(allowed):
            os.sched_setaffinity(0, cpus)
            return "bound to %d CPUs local to GPU %d (%d-%d)" % (len(cpus), index, min(cpus), max(cpus))
        return "all %d CPUs are local to GPU %d" % (len(allowed), index)
    except Exception as e:  # no NVML / not permitted: run unbound
        return "unbound (%s)" % type(e).__name__


def _synth_frame_torch(torch, synth, width, height, t, seed):
    """slowflow_b200.synth.frame (SURVEY 8d recipe) in float64 on the current CUDA device -> float32 (3, H, W)."""
    dev = torch.device("cuda")
    y = torch.arange(height, dtype=torch.float64, device=dev)[:, None].expand(height, width)
    x = torch.arange(width, dtype=torch.float64, device=dev)[None, :].expand(height, width)
    pi = 3.141592653589793
    u = 1.0 + 2.0 * torch.sin(2 * pi * y / height * 1.5) + (x > width / 2).to(torch.float64) * 3.0
    v = 1.5 * torch.cos(2 * pi * x / width * 2)
    xs, ys = x - t * u, y - t * v
    theta, phi = synth.texture_params(seed)
    out = torch.full((3, height, width), 127.5, dtype=torch.float64, device=dev)
    for k, (lam, amp) in enumerate(zip(synth._WAVELENGTHS, synth._AMPLITUDES)):
        arg = (2 * pi / lam) * (xs * float(__import__("math").cos(theta[k])) + ys * float(__import__("math").sin(theta[k])))
        for c in range(3):
            out[c] += amp * 0.68 * torch.sin(arg + float(phi[c, k]))
    return out.to(torch.float32)


# ----------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    # one WHOLE field per host core and step (variational.c:101 on the full 2560x1440 pair; the reference's own
    # parallel model is one window per core, slow_flow.cpp:706): ~6 s per step
    runner = CpuOracleRunner(args.width, args.height, args.height, cores)
    kind, sample = runner.kind, runner.sample
    vals = []
    for i in range(args.warmup + args.steps):
        f, dt = runner.step()
        if i >= args.warmup:
            vals.append((f, dt))
    runner.close()
    tot_t = sum(d for _, d in vals)
    fields = sum(f for f, _ in vals)
    value = fields / tot_t
    line = {
        "impl": "reference", "metric": "refined_flow_fields_per_sec_2560x1440", "value": value, "unit": "fields/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, len(vals)),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD % (args.width, args.height), "fields_per_step": cores,
                   "parallelism": "cpu: one whole field per host core (reference model: omp parallel for over windows)"},
        "cpu_baseline": {"value": value, "unit": "fields/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "fields/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------- multi-frame secondary
MT_BYTES_PER_PX_OUTER = 1468.0  # fully fused streaming model of one outer iteration at S=3 (SURVEY 8d)


def _mt_params(layers):
    """BASELINE config 3 / 4 parameters (SURVEY 8d): S=3, Geman-McClure eps 0.5 colour penalty, occlusion reasoning,
    2 alternations x 10 outer x 1 inner x 30 SOR sweeps, thresholds 1e-5, 8-bit intensities."""
    from slowflow_b200 import mt_params_default
    p = mt_params_default()
    p.S, p.hbit, p.layers = 3, 0, layers
    p.niter_alter, p.niter_outer = 2, 10
    p.robust_color, p.robust_color_eps = 4, 0.5
    return p


def run_mt_secondary(ctx, torch, with_cpu, reps=3):
    """Times sfgpu_variational_mt (host-buffer C ABI: uploads, pyramid, occlusion labelling and downloads included) on
    one synthetic window of BASELINE config 3 (1280x1024) and config 4 (2560x1440, 3 pyramid layers, zero initial flow).
    with_cpu: the reference's own CPU driver (oracle/_ref, lexicographic SOR, one core) on a bounded sample of the same
    window -- 1 alternation x 2 (config 3) / x 1 (config 4) outer iterations per level -- as seconds per outer iteration."""
    import ctypes as C
    import numpy as np
    from slowflow_b200 import ColorImage, Image, synth
    from slowflow_b200.image import color_image_t
    from slowflow_b200.params import MTParams
    peak, _ = measured_peak_gbs()
    out = {}
    for cid, (w, h, layers, zero) in ((3, (1280, 1024, 1, False)), (4, (2560, 1440, 3, True))):
        S4 = ((w + 3) // 4) * 4
        P = S4 * h
        pins = [torch.empty(3 * P, dtype=torch.float32).pin_memory() for _ in range(5)]
        frames = []
        for k, t in enumerate(range(-2, 3)):
            ci = ColorImage(w, h, buffer=pins[k].numpy())
            ci.array[:] = _synth_frame_torch(torch, synth, w, h, t, 20170721).cpu().numpy()
            frames.append(ci)
        raw = [f.copy() for f in frames] if with_cpu else None
        u0, v0 = synth.initial_flow(w, h, zero=zero)
        p = _mt_params(layers)
        q = MTParams.from_buffer_copy(bytes(p))
        ctx.normalize(frames, q)
        pin_x, pin_y = torch.empty(P, dtype=torch.float32).pin_memory(), torch.empty(P, dtype=torch.float32).pin_memory()
        wx, wy = Image(w, h, buffer=pin_x.numpy()), Image(w, h, buffer=pin_y.numpy())
        times, stats, prof = [], None, None
        for rep in range(reps + 1):
            wx.array[:] = u0
            wy.array[:] = v0
            ctx.profile_enable(True)
            ctx.profile_reset()
            ctx.synchronize()
            t0 = time.perf_counter()
            ctx.variational_mt(wx, wy, frames, q, None, None)
            dt = time.perf_counter() - t0
            pr = ctx.profile_get()
            if rep > 0:
                times.append(dt)
                stats, prof = ctx.mt_stats(), pr
        ctx.profile_enable(False)
        times.sort()
        t_win = times[len(times) // 2]
        model_bytes = MT_BYTES_PER_PX_OUTER * stats.pixel_outer_iterations
        host_ms = stats.setup_ms + stats.graphcut_ms + prof.graphcut_ms
        line = {
            "workload": "Variational_MT %dx%d, S=3 (5 frames), %d pyramid layer(s), Geman-McClure eps 0.5, occlusion reasoning, "
                        "2 alternations x 10 outer x 1 inner x 30 SOR, %s initial flow (BASELINE config %d)"
                        % (w, h, layers, "zero" if zero else "noisy", cid),
            "ms_per_window": 1e3 * t_win, "windows_per_sec": 1.0 / t_win, "reps": reps, "levels": stats.levels,
            "outer_iterations_executed": stats.outer_iterations, "sor_calls": stats.sor_calls,
            "graphcut_calls": stats.graphcut_calls, "ms_per_outer_iteration": 1e3 * t_win / max(1, stats.outer_iterations),
            "split_ms": {"upload_and_pyramid": stats.setup_ms, "occlusion_labelling_device": prof.graphcut_ms,
                         "occlusion_labelling_host": stats.graphcut_ms,
                         "sor_kernels": prof.sor_ms, "data_term_kernels": prof.data_ms,
                         "other": max(0.0, stats.total_ms - host_ms - prof.sor_ms - prof.data_ms), "total_in_library": stats.total_ms},
            "kernel_launches": int(prof.kernel_launches),
            "data_term_launches_per_outer_iteration": prof.data_launches / max(1, stats.outer_iterations),
            "fused_model": {"bytes_per_px_per_outer_iteration": MT_BYTES_PER_PX_OUTER, "bytes": model_bytes,
                            "achieved_gbs": model_bytes / t_win / 1e9, "frac": model_bytes / t_win / 1e9 / peak, "peak_gbs": peak},
            "api": "sfgpu_variational_mt (host pinned buffers, H2D/D2H inside the timed region)",
        }
        if with_cpu:
            from oracle.pyoracle import Reference, have_reference, Oracle
            lib, prefix, kind = (Reference().lib, "sf_ref_", "reference") if have_reference() else (Oracle().lib, "sfo_", "port")
            n_outer = 2 if cid == 3 else 1
            pc = _mt_params(layers)
            pc.niter_alter, pc.niter_outer = 1, n_outer
            CP = C.POINTER(color_image_t)
            arr = (CP * 5)(*[C.pointer(f.c) for f in raw])
            cx, cy, occ = Image.from_array(u0), Image.from_array(v0), Image(w, h)
            avg, st = (C.c_float * 2)(), (C.c_int * 2)()
            with _StdoutToStderr():
                t0 = time.perf_counter()
                getattr(lib, prefix + "normalize")(arr, 5, C.byref(pc))
                getattr(lib, prefix + "variational_mt")(cx.ptr(), cy.ptr(), arr, C.byref(pc), None, occ.ptr(), avg, 0, st)
                cpu_s = time.perf_counter() - t0
            per_outer_cpu = cpu_s / (n_outer * layers)
            line["cpu_baseline"] = {
                "value": per_outer_cpu, "unit": "s per outer iteration (1 core)", "cores": 1, "kind": kind,
                "sample": "normalize + 1 alternation x %d outer iteration(s) per level of the same window, lexicographic SOR, "
                          "%.1f s of CPU" % (n_outer, cpu_s),
                "gpu_ms_per_outer_iteration": 1e3 * t_win / max(1, stats.outer_iterations)}
        out["config%d" % cid] = line
        del pins, frames
    out["epic"] = run_epic_secondary(ctx, with_cpu)
    out["config5_mt_driver"] = run_driver_secondary()
    return out


def run_driver_secondary(w=1280, h=1024, jets=8, S=3):
    """BASELINE config 5, secondary: the synthetic sequence as multi-frame windows (forward AND backward solve per jet,
    slow_flow.cpp:875-1030) through the compiled sharded driver (tools/slow_flow_gpu.cpp -> slowflow_b200/lib/slow_flow_gpu):
    PPM frames in, .flo / _back.flo / occlusion .pbm out, with 1 and 2 host threads per GPU.  The window loop's own clock
    (frame loading and normalize() excluded, result writing included)."""
    import re
    import subprocess
    import tempfile
    import numpy as np
    from slowflow_b200 import synth
    exe = os.path.join(ROOT, "slowflow_b200", "lib", "slow_flow_gpu")
    if not os.path.exists(exe):
        return {"unavailable": "slowflow_b200/lib/slow_flow_gpu is not built"}
    steps = S - 1
    n = 1 + (jets + 2) * steps
    res = {"workload": "%d jets (= %d Variational_MT windows) of a %d-frame synthetic %dx%d PPM sequence, S=%d, config-3 parameters, "
                       "results written to a temporary directory" % (jets, 2 * jets, n, w, h, S),
           "api": "slow_flow_gpu (sharded window driver, one or two host threads per device)"}
    try:
        with tempfile.TemporaryDirectory() as d:
            for k in range(n):
                f = np.clip(np.rint(synth.frame(w, h, k - steps)), 0, 255).astype(np.uint8)
                with open(os.path.join(d, "frame_%d.ppm" % k), "wb") as fh:
                    fh.write(b"P6\n%d %d\n255\n" % (w, h))
                    fh.write(np.ascontiguousarray(f.transpose(1, 2, 0)).tobytes())
            for tpg in (1, 2):
                r = subprocess.run([exe, "--frames", os.path.join(d, "frame_%d.ppm"), "--out", os.path.join(d, "out%d" % tpg), "--start", str(steps),
                                    "--jets", str(jets), "--S", str(S), "--gpus", "1", "--threads-per-gpu", str(tpg), "--occlusions",
                                    "--set", "slow_flow_occlusion_reasoning=1", "--set", "slow_flow_niter_alter=2",
                                    "--set", "slow_flow_robust_color=4", "--set", "slow_flow_robust_color_eps=0.5", "--set", "16bit=0",
                                    "--set", "slow_flow_smoothing=1", "--set", "slow_flow_omega_0=0", "--set", "slow_flow_omega_1=2",
                                    "--set", "slow_flow_occlusion_penalty=0.1", "--set", "slow_flow_occlusion_alpha=0.1"],
                                   capture_output=True, text=True, timeout=300)
                m = re.search(r"window loop: ([0-9.]+) s, ([0-9.]+) jets/s", r.stdout)
                if r.returncode != 0 or not m:
                    res["threads_per_gpu_%d" % tpg] = {"error": (r.stderr or r.stdout)[-200:]}
                    continue
                res["threads_per_gpu_%d" % tpg] = {"window_loop_s": float(m.group(1)), "jets_per_sec": float(m.group(2)),
                                                   "windows_per_sec": 2.0 * float(m.group(2))}
    except Exception as e:  # the secondary must never take the bench line down
        res["error"] = repr(e)[:200]
    return res


def run_epic_secondary(ctx, with_cpu, reps=3):
    """EPIC sparse-to-dense interpolation (the step in front of variational(), epicflow.cpp:125): sfgpu_epic on synthetic
    matches / edge costs at 1024x436 (5,000 matches, the EpicFlow paper's Sintel geometry) and 2560x1440 (20,000 matches),
    host buffers in, flow planes out; with_cpu: the reference's own epic() (oracle/_ref, one core) on the same inputs."""
    import ctypes as C
    import numpy as np
    from slowflow_b200 import ColorImage, Image, synth
    from slowflow_b200.api import EpicParams, epic_params_default
    from slowflow_b200.image import color_image_t, image_t
    out = {}
    for (w, h, n) in ((1024, 436, 5000), (2560, 1440, 20000)):
        im, m, edges = synth.epic_case(w, h, n)
        ci = ColorImage.from_array(im)
        p = epic_params_default()
        fx, fy = Image(w, h), Image(w, h)
        times, st = [], None
        for rep in range(reps + 1):
            e = edges.copy()
            ctx.synchronize()
            t0 = time.perf_counter()
            st = ctx.epic(fx, fy, ci, m, e, p)
            dt = time.perf_counter() - t0
            if rep > 0:
                times.append(dt)
        times.sort()
        line = {"workload": "EPIC interpolation %dx%d, %d synthetic matches, LA fit, default parameters" % (w, h, n),
                "ms_per_call": 1e3 * times[len(times) // 2], "matches_after_filters": st.matches_after_consistency,
                "distance_transform_sweeps": [st.sweeps_prefilter, st.sweeps_interpolation],
                "api": "sfgpu_epic (host buffers, uploads and the flow download inside the timed region)"}
        if with_cpu:
            from oracle.pyoracle import Reference, have_reference
            if have_reference():
                L = Reference().lib
                IP, CP = C.POINTER(image_t), C.POINTER(color_image_t)
                L.sf_ref_epic.argtypes = [IP, IP, CP, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(EpicParams)]
                L.sf_ref_epic.restype = None
                rx, ry, e = Image(w, h), Image(w, h), edges.copy()
                with _StdoutToStderr():
                    t0 = time.perf_counter()
                    L.sf_ref_epic(rx.ptr(), ry.ptr(), ci.ptr(), m.ctypes.data, n, 4, e.ctypes.data, C.byref(p))
                    cpu_s = time.perf_counter() - t0
                d = np.sqrt((fx.array - rx.array) ** 2 + (fy.array - ry.array) ** 2)
                line["cpu_baseline"] = {"value": cpu_s, "unit": "s per call (1 core)", "cores": 1, "kind": "reference",
                                        "sample": "the same call through the reference's epic() (sgels from oracle/ref_glue/lapack_stub.c)",
                                        "gpu_vs_cpu_mean_px": float(d.mean()), "gpu_vs_cpu_max_px": float(d.max())}
        out["%dx%d" % (w, h)] = line
    return out


# ----------------------------------------------------------------------------------------- our arm
DUMP_SAMPLES = 1 << 21  # per flow component when the whole output exceeds DUMP_LIMIT_BYTES: 32 MB in all with the index
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, d_wx, d_wy, W, H, S):
    """What a caller of sfgpu_variational_dev receives from one step: the refined flow of every pair, cropped from the row stride
    S to the image width, as float32 flow_x.npy / flow_y.npy of shape (pairs, H, W).  When the two exceed DUMP_LIMIT_BYTES, the
    same fixed, seeded sample of (pair, row, column) positions is taken from both instead (1-D arrays), and the positions'
    indices into the (pairs, H, W) array go to sample_index.npy (float64, exact below 2**53).  The inputs depend only on the
    arguments, so two builds run with the same arguments can be compared file for file."""
    import numpy as np
    import torch
    B = len(d_wx)
    n = B * H * W
    fx = torch.stack(d_wx).view(B, H, S)[:, :, :W]
    fy = torch.stack(d_wy).view(B, H, S)[:, :, :W]
    if 2 * 4 * n <= DUMP_LIMIT_BYTES:
        out = {"flow_x": fx.cpu().numpy(), "flow_y": fy.cpu().numpy()}
    else:
        idx = np.unique(np.random.default_rng(20170721).integers(0, n, size=DUMP_SAMPLES))
        ti = torch.from_numpy(idx).to(fx.device)
        out = {"flow_x": fx.reshape(-1)[ti].cpu().numpy(), "flow_y": fy.reshape(-1)[ti].cpu().numpy(),
               "sample_index": idx.astype(np.float64)}
    os.makedirs(dirname, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def _profile_counts():
    """Per-launch counters of the kernels from the committed ncu --set full capture (profiles/kernel_counts.json):
    evidence of the build that was profiled, reported under `from_profile`, never presented as measured in this run."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "kernel_counts.json")))
    except Exception:
        return {}


def _data_term_roofline(prof, peak_gbs, pixels, clocks_mhz, counts):
    """Second kernel of the path (k_prep_two_frame: warp + derivatives + data term + Laplacian + block inverse): HBM ceiling
    (52 B/px algorithmic, SURVEY 8d) from the live CUDA-event time; the issue-slot ceiling uses the warp-instruction count
    of the committed ncu capture (scaled by pixels) and the SM clock sampled during this run."""
    if prof.data_ms <= 0 or prof.data_launches <= 0:
        return None
    t = prof.data_ms * 1e-3 / prof.data_launches
    gbs = DATA_BYTES_PER_PX * prof.data_pixels / (prof.data_ms * 1e-3) / 1e9
    r = {"kernel": "k_prep_two_frame", "bound": "hbm", "achieved": gbs, "peak": peak_gbs, "unit": "GB/s", "frac": gbs / peak_gbs,
         "avg_launch_ms": t * 1e3, "launches": int(prof.data_launches),
         "algorithmic_bytes_per_launch": DATA_BYTES_PER_PX * pixels,
         "hbm_bound_ms": DATA_BYTES_PER_PX * pixels / (peak_gbs * 1e9) * 1e3}
    c = counts.get("k_prep_two_frame")
    if c and clocks_mhz:
        warp_inst = float(c["warp_instructions_per_launch"]) / float(c["pixels"]) * pixels
        issue_s = warp_inst / (148 * 4 * clocks_mhz * 1e6)
        r["from_profile"] = {"source": c.get("source"), "warp_instructions_per_launch": warp_inst,
                             "dram_bytes_per_launch": c.get("dram_bytes_per_launch"),
                             "issue_bound_ms": issue_s * 1e3, "issue_frac": issue_s / t, "sm_clock_mhz_this_run": clocks_mhz}
    return r


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from slowflow_b200 import ColorImage, Context, Image, synth, variational, variational_params_default
    from slowflow_b200.shard import max_over_ranks, shard_range, sum_over_ranks

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the GPU path has no CPU fallback")
    torch.cuda.set_device(local)
    affinity = _bind_to_gpu_numa_node(local)  # before any pinned allocation (first touch decides the NUMA node)
    if world > 1:
        # rank 0 prints ONE JSON line on stdout: NCCL's version banner and warnings (NCCL_DEBUG=VERSION/WARN/INFO write to
        # stdout by default) go to stderr instead
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":  # this level printf()s its banner straight to stdout
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    W, H, B = args.width, args.height, args.pairs
    first_frame, scaling = 0, "weak"
    if args.total_pairs > 0:
        # strong scaling: one sequence, rank r refines the contiguous pair range shard_range gives it (a frame shared by
        # two pairs of the same rank is uploaded once; the frame at a range boundary is uploaded by both neighbours)
        lo, hi = shard_range(args.total_pairs, rank, world)
        first_frame, B, scaling = lo, hi - lo, "strong"
        if B < 1:
            raise SystemExit("bench.py: --total-pairs must be at least the number of ranks")
    S = ((W + 3) // 4) * 4
    P = S * H
    params = variational_params_default()

    # ---- synthetic window of B+1 consecutive frames (rank-specific texture seed) + initial flow.  The frames are 8-bit
    # images (the analytic texture rounded to integers, like the camera frames adaptiveFR.cpp:450-464 loads); they exist
    # twice in pinned host memory: packed interleaved u8 (H, W, 3) and as the planar fp32 images mat2colorImg makes of them
    seed = 20170721 + (1000 * rank if scaling == "weak" else 0)
    host_frames = [torch.empty(3 * P, dtype=torch.float32).pin_memory() for _ in range(B + 1)]
    host_u8 = [torch.empty((H, W, 3), dtype=torch.uint8).pin_memory() for _ in range(B + 1)]
    frames = []
    for t in range(B + 1):
        ci = ColorImage(W, H, buffer=host_frames[t].numpy())
        # the analytic texture of slowflow_b200.synth evaluated with torch on the device (set-up only: 2 s per
        # frame with numpy), then parked in pinned HOST memory -- the timed e2e region uploads it again
        f = torch.clamp(torch.round(_synth_frame_torch(torch, synth, W, H, first_frame + t, seed)), 0, 255)
        ci.array[:] = f.cpu().numpy()
        host_u8[t].copy_(f.permute(1, 2, 0).to(torch.uint8).cpu())
        frames.append(ci)
    frames_u8 = [t.numpy() for t in host_u8]
    if rank == 0:
        yy, xx = np.mgrid[0:8, 0:W].astype(np.float64)
        gu, gv = synth.gt_flow(W, H)
        chk = synth.texture(xx - (first_frame + 1) * gu[:8], yy - (first_frame + 1) * gv[:8], seed).astype(np.float32)
        if not np.allclose(frames[1].array[:, :8, :], np.clip(np.rint(chk), 0, 255), atol=1.001):
            raise SystemExit("bench.py: device-generated synthetic frame differs from slowflow_b200.synth")
    u0, v0 = synth.initial_flow(W, H)
    init_x, init_y = Image.from_array(u0), Image.from_array(v0)
    host_wx = [torch.empty(P, dtype=torch.float32).pin_memory() for _ in range(B)]
    host_wy = [torch.empty(P, dtype=torch.float32).pin_memory() for _ in range(B)]
    wxs = [Image(W, H, buffer=t.numpy()) for t in host_wx]
    wys = [Image(W, H, buffer=t.numpy()) for t in host_wy]

    stream = torch.cuda.Stream()
    ctx = Context(local, stream=stream.cuda_stream)
    ctx.set_sor_variant(args.sor_variant)
    ctx.set_sor_fuse(args.sor_fuse)

    # ---- device-resident copies for `value`
    d_frames = [f.cuda(non_blocking=True) for f in host_frames]
    d_init_x = torch.from_numpy(init_x.buf.copy()).cuda()
    d_init_y = torch.from_numpy(init_y.buf.copy()).cuda()
    d_wx = [torch.empty(P, dtype=torch.float32, device="cuda") for _ in range(B)]
    d_wy = [torch.empty(P, dtype=torch.float32, device="cuda") for _ in range(B)]
    torch.cuda.synchronize()

    def step_resident():
        with torch.cuda.stream(stream):
            for j in range(B):
                d_wx[j].copy_(d_init_x, non_blocking=True)
                d_wy[j].copy_(d_init_y, non_blocking=True)
                ctx.variational_dev(d_wx[j].data_ptr(), d_wy[j].data_ptr(), d_frames[j].data_ptr(),
                                    d_frames[j + 1].data_ptr(), W, H, S, params)

    def reset_host_flows():
        for j in range(B):
            wxs[j].buf[:] = init_x.buf
            wys[j].buf[:] = init_y.buf

    def step_e2e():
        # wx, wy are in/out like in the reference (variational.c:68-69): later steps refine the previous
        # step's output; the work per step is identical (no data-dependent control flow on this path)
        ctx.variational_sequence_int(frames_u8, wxs, wys, params)

    def step_e2e_f32():
        ctx.variational_sequence(frames, wxs, wys, params)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_host(fn, steps):
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        return max_over_ranks(time.perf_counter() - t0)

    # ---- warm-up (all paths), then the device-resident timed region
    for _ in range(args.warmup):
        step_resident()
    reset_host_flows()
    step_e2e_f32()
    barrier()
    same_f32 = bool(np.array_equal(d_wx[0].cpu().numpy(), wxs[0].buf))
    reset_host_flows()
    step_e2e()
    barrier()
    # parity spot check of the timed paths (not timed): pair 0 resident == pair 0 through the host ABI (u8 and fp32 frames)
    same = bool(np.array_equal(d_wx[0].cpu().numpy(), wxs[0].buf)) and same_f32
    reset_host_flows()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # ---- timed region 1 (the metric): exactly K steps, nothing but the library's own launches on the stream
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step_resident()
    e1.record(stream)
    barrier()
    ms_plain = e0.elapsed_time(e1)
    ms = max_over_ranks(ms_plain)
    total_fields = sum_over_ranks(B * args.steps)
    value = total_fields / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_wx, d_wy, W, H, S)
    # ---- timed region 2 (kernel attribution): the same K steps with CUDA events around every sor_coupled call and
    # every data-term launch.  Kept out of region 1 because an event record between two launches breaks their
    # programmatic-dependent-launch chaining (sf_internal.cuh: pdl_enter), i.e. it perturbs what it measures.
    ctx.profile_enable(True)
    ctx.profile_reset()
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step_resident()
    e1.record(stream)
    barrier()
    ms_local = e0.elapsed_time(e1)
    prof = ctx.profile_get()
    ctx.profile_enable(False)
    ctx.profile_reset()

    # ---- end-to-end through the host-buffer ABI (H2D + D2H inside the timed region): 8-bit frames (headline), fp32 frames
    e2e_s = timed_host(step_e2e, args.steps)
    launches_e2e = int(ctx.profile_get().kernel_launches)
    clocks = sampler.stop() if rank == 0 else None
    e2e_value = total_fields / e2e_s
    h2d = 3 * W * H * (B + 1) + 2 * P * B * 4
    d2h = 2 * P * B * 4
    f32_steps = max(1, min(args.steps, 5))
    e2e_f32_s = timed_host(step_e2e_f32, f32_steps)
    h2d_f32 = (3 * P * (B + 1) + 2 * P * B) * 4

    # ---- the UNMODIFIED drop-in call: variational() (variational.h:30) on ordinary malloc'ed buffers, one pair per call,
    # synchronous, exactly what adaptiveFR.cpp:574 / epicflow.cpp:127 would execute after re-linking
    n_legacy = min(6, B)
    lg_frames = [ColorImage.from_array(frames[k].array) for k in range(n_legacy + 1)]  # numpy memory: pageable
    lg_x, lg_y = [Image.from_array(u0) for _ in range(n_legacy)], [Image.from_array(v0) for _ in range(n_legacy)]
    torch.cuda.synchronize()
    variational(Image.from_array(u0), Image.from_array(v0), lg_frames[0], lg_frames[1], None)  # creates the thread's default context
    legacy_s = timed_host(lambda: [variational(lg_x[j], lg_y[j], lg_frames[j], lg_frames[j + 1], None) for j in range(n_legacy)], 1)
    legacy_same = bool(np.array_equal(lg_x[0].array, d_wx[0].cpu().numpy().reshape(H, S)[:, :W]))

    # ---- roofline of the dominant kernel (SOR)
    peak, peak_src = measured_peak_gbs()
    counts = _profile_counts()
    sor_bytes = SOR_BYTES_PER_PX_SWEEP * prof.sor_pixel_sweeps
    sor_gbs = sor_bytes / (prof.sor_ms * 1e-3) / 1e9 if prof.sor_ms > 0 else 0.0
    fuse = args.sor_fuse or 4  # sf_context.cu: auto_fuse
    sor_launch_s = prof.sor_ms * 1e-3 / max(1, prof.sor_launches)
    # dram__bytes_read.sum + dram__bytes_write.sum per k_sor_tiled launch: from the committed ncu --set full capture of the
    # profiled build (profiles/kernel_counts.json), divided by THIS run's live launch time
    sc = counts.get("k_sor_tiled") or {}
    traffic = sc.get("dram_bytes_per_launch") if (W, H) == (W_FULL, H_FULL) else None
    roofline = {
        "bound": "hbm", "kernel": "k_sor_tiled (red-black SOR, %d sweeps per pass over the image, all passes of a call chained in one launch)" % fuse,
        "achieved": sor_gbs, "peak": peak, "unit": "GB/s", "frac": sor_gbs / peak, "traffic": traffic,
        "peak_source": peak_src,
        "algorithmic_bytes_per_launch": sor_bytes / max(1, prof.sor_launches),
        "avg_launch_ms": 1e3 * sor_launch_s, "launches": int(prof.sor_launches),
        "sor_share_of_step": prof.sor_ms / ms_local if ms_local > 0 else None,
        "instrumented_ms_per_step": ms_local / args.steps,
        # what the DRAM really moved (ncu, per launch, profiled build) over the live launch time: temporal blocking makes
        # it ~4x smaller than the algorithmic figure, so `frac` above can exceed 1 while the HBM interface is half busy
        "from_profile": {"source": sc.get("source"), "dram_bytes_per_launch": traffic,
                         "dram_achieved_gbs": (traffic / sor_launch_s / 1e9) if traffic and sor_launch_s > 0 else None,
                         "dram_frac": (traffic / sor_launch_s / 1e9 / peak) if traffic and sor_launch_s > 0 else None},
        "data_term": _data_term_roofline(prof, peak, W * H, (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz"), counts),
    }

    line = {
        "metric": "refined_flow_fields_per_sec_2560x1440", "value": value, "unit": "fields/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD % (W, H), "fields_per_step": sum_over_ranks(B),
                   "pairs_per_gpu_per_step": B, "parallelism": "independent consecutive frame pairs per GPU (config 5 sharding), no collective",
                   "host_affinity": affinity,
                   "l2": "per-pair working set %.0f MB > 126 MB L2 (no flush needed)" % (26 * P * 4 / 1e6),
                   "sor": "red-black, variant %d, fuse %d" % (args.sor_variant, fuse)},
        "e2e": {"value": e2e_value, "unit": "fields/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "sfgpu_variational_sequence_u8 (8-bit frames + fp32 flows in pinned host memory)",
                "matches_resident_result": same,
                "host_gbs": {"h2d": world * h2d * args.steps / e2e_s / 1e9, "d2h": world * d2h * args.steps / e2e_s / 1e9,
                             "note": "whole job, all ranks"},
                "f32_frames": {"value": sum_over_ranks(B * f32_steps) / e2e_f32_s, "unit": "fields/s", "steps": f32_steps,
                               "h2d_bytes_per_step": h2d_f32, "d2h_bytes_per_step": d2h,
                               "api": "sfgpu_variational_sequence (fp32 frames in pinned host memory)"},
                "legacy": {"value": sum_over_ranks(n_legacy) / legacy_s, "unit": "fields/s", "pairs": n_legacy,
                           "ms_per_call": 1e3 * legacy_s / n_legacy, "matches_resident_result": legacy_same,
                           "api": "variational() (variational.h:30), one synchronous call per pair on pageable malloc'ed images"}},
        "gpu_launches": int(prof.kernel_launches),
        "gpu_launches_e2e": launches_e2e,
        "roofline": roofline,
        "clocks": clocks,
    }
    if rank == 0 and world == 1 and not args.no_secondary:
        # the resident buffers of the two-frame legs are not needed any more
        del d_frames, d_wx, d_wy, host_frames, host_u8, frames, frames_u8
        torch.cuda.empty_cache()
        line["secondary"] = run_mt_secondary(ctx, torch, with_cpu=not args.no_cpu_baseline)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        runner = CpuOracleRunner(W, H, H, 1)
        f, dt = runner.step()
        line["cpu_baseline"] = {"value": f / dt, "unit": "fields/s", "cores": 1, "kind": runner.kind,
                                "sample": runner.sample,
                                "host_cores_available": os.cpu_count()}
    if rank == 0:
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    a = parse()
    sys.exit(run_reference(a) if a.impl == "reference" else run_ours(a))
