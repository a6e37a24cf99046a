"""Host-side mirror of the reference entry points over the C ABI (include/slowflow_gpu.h).

``variational(wx, wy, im1, im2, params)``   -> epic_flow_extended/variational.c:101
``Variational_MT().variational(wx, wy, im, params)`` -> epic_flow_extended/variational_mt.cpp:526
``Context`` wraps an ``sfgpu_ctx`` handle (one per host thread / device / stream).

All compute goes through ``libslowflow_gpu.so``; a missing library or GPU raises ``RuntimeError``.
"""
import ctypes as C
import os

from .image import Image, ColorImage, image_t, color_image_t
from .params import VariationalParams, MTParams, mt_params_default

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def library_path():
    """Path of the CUDA library; SLOWFLOW_GPU_LIB overrides it (used to A/B kernel build variants)."""
    return os.environ.get("SLOWFLOW_GPU_LIB") or os.path.join(_HERE, "lib", "libslowflow_gpu.so")


class Profile(C.Structure):
    _fields_ = [("sor_ms", C.c_double), ("sor_launches", C.c_longlong), ("sor_calls", C.c_longlong),
                ("sor_pixel_sweeps", C.c_longlong), ("data_ms", C.c_double), ("data_launches", C.c_longlong),
                ("data_pixels", C.c_longlong), ("kernel_launches", C.c_longlong), ("graphcut_ms", C.c_double)]


class FrameInt(C.Structure):
    """sf_frame_int_t: the cv::Mat fields of an 8-/16-bit frame (include/slowflow_gpu.h)."""
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("channels", C.c_int), ("step", C.c_size_t),
                ("data", C.c_void_p)]


class EpicParams(C.Structure):
    """epic_params_t (epic_flow_extended/epic.h:5-14)."""
    _fields_ = [("method", C.c_char * 20), ("saliency_th", C.c_float), ("pref_nn", C.c_int), ("pref_th", C.c_float),
                ("nn", C.c_int), ("coef_kernel", C.c_float), ("euc", C.c_float), ("verbose", C.c_int)]


class FloatImage(C.Structure):
    """float_image (array_types.h:70-77): row-major tx columns x ty rows."""
    _fields_ = [("pixels", C.POINTER(C.c_float)), ("tx", C.c_int), ("ty", C.c_int)]


class EpicStats(C.Structure):
    _fields_ = [("matches_in", C.c_int), ("matches_after_saliency", C.c_int), ("matches_after_consistency", C.c_int),
                ("sweeps_prefilter", C.c_int), ("sweeps_interpolation", C.c_int)]


class MTStats(C.Structure):
    _fields_ = [("levels", C.c_int), ("outer_iterations", C.c_int), ("sor_calls", C.c_int),
                ("graphcut_calls", C.c_int), ("setup_ms", C.c_double), ("graphcut_ms", C.c_double),
                ("total_ms", C.c_double), ("pixel_outer_iterations", C.c_longlong)]


# every symbol include/slowflow_gpu.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "variational_params_default", "variational", "sf_mt_params_default", "sfgpu_create", "sfgpu_destroy",
    "sfgpu_last_error", "sfgpu_device_count", "sfgpu_synchronize", "sfgpu_set_sor_variant", "sfgpu_set_sor_fuse",
    "sfgpu_variational", "sfgpu_variational_dev", "sfgpu_variational_sequence", "sfgpu_variational_sequence_u8",
    "sfgpu_variational_sequence_u16", "sfgpu_host_register",
    "sfgpu_host_unregister", "sfgpu_variational_mt", "sfgpu_mt_frame_cache", "sfgpu_normalize", "sfgpu_get_mt_stats", "sfgpu_profile_enable",
    "sfgpu_profile_reset", "sfgpu_profile_get", "sfgpu_image_warp", "sfgpu_warp_frame_derivs", "sfgpu_compute_dpsis_weight",
    "sfgpu_compute_smoothness", "sfgpu_compute_data_and_match", "sfgpu_prep_two_frame", "sfgpu_mt_system", "sfgpu_mt_occ_costs", "sfgpu_sub_laplacian", "sfgpu_sor_coupled",
    "sfgpu_epic", "sfgpu_epic_batch", "sfgpu_epic_nnfield", "sfgpu_rgb_to_lab", "sfgpu_epicflow_sequence", "epic_params_default", "sfgpu_version", "sfgpu_grid_mincut", "sfgpu_grid_mincut_dev", "sfgpu_prescale_size", "sfgpu_prescale", "sfgpu_raw_weighting",
    "sfgpu_write_flo", "sfgpu_read_flo_size", "sfgpu_read_flo", "sfgpu_write_occlusion_pbm", "sfgpu_set_device", "sfgpu_get_device",
    "sfgpu_convolve_horiz", "sfgpu_convolve_vert", "sfgpu_color_image_convolve_hv", "sfgpu_get_derivatives",
]


def load_library(path=None):
    """dlopen the CUDA library (RTLD_LOCAL: it exports ``variational`` like the reference does)."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    p = path or library_path()
    if not os.path.exists(p):
        raise RuntimeError(
            "libslowflow_gpu.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'`. "
            "There is no CPU fallback." % p)
    lib = C.CDLL(p, mode=os.RTLD_LOCAL | os.RTLD_NOW)
    IP, CP, VP = C.POINTER(image_t), C.POINTER(color_image_t), C.POINTER(VariationalParams)
    FP = C.POINTER(C.c_float)
    lib.sfgpu_last_error.restype = C.c_char_p
    lib.sfgpu_version.restype = C.c_char_p
    lib.sfgpu_create.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
    lib.sfgpu_destroy.argtypes = [C.c_void_p]
    lib.sfgpu_destroy.restype = None
    lib.sfgpu_synchronize.argtypes = [C.c_void_p]
    lib.sfgpu_set_sor_variant.argtypes = [C.c_void_p, C.c_int]
    lib.sfgpu_set_sor_fuse.argtypes = [C.c_void_p, C.c_int]
    lib.variational_params_default.argtypes = [VP]
    lib.variational_params_default.restype = None
    lib.variational.argtypes = [IP, IP, CP, CP, VP]
    lib.variational.restype = None
    lib.sf_mt_params_default.argtypes = [C.POINTER(MTParams)]
    lib.sf_mt_params_default.restype = None
    lib.sfgpu_variational.argtypes = [C.c_void_p, IP, IP, CP, CP, VP]
    lib.sfgpu_variational_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                          C.c_int, C.c_int, VP]
    lib.sfgpu_variational_sequence.argtypes = [C.c_void_p, C.c_int, C.POINTER(CP), C.POINTER(IP), C.POINTER(IP), VP]
    for name in ("sfgpu_variational_sequence_u8", "sfgpu_variational_sequence_u16"):
        getattr(lib, name).argtypes = [C.c_void_p, C.c_int, C.POINTER(FrameInt), C.POINTER(IP), C.POINTER(IP), VP, C.c_int]
    lib.sfgpu_host_register.argtypes = [C.c_void_p, C.c_ulonglong]
    lib.sfgpu_host_unregister.argtypes = [C.c_void_p]
    lib.sfgpu_variational_mt.argtypes = [C.c_void_p, IP, IP, C.POINTER(CP), C.POINTER(MTParams), CP, IP, FP]
    lib.sfgpu_normalize.argtypes = [C.c_void_p, C.POINTER(CP), C.c_int, C.POINTER(MTParams)]
    lib.sfgpu_get_mt_stats.argtypes = [C.c_void_p, C.POINTER(MTStats)]
    lib.sfgpu_profile_enable.argtypes = [C.c_void_p, C.c_int]
    lib.sfgpu_profile_reset.argtypes = [C.c_void_p]
    lib.sfgpu_profile_get.argtypes = [C.c_void_p, C.POINTER(Profile)]
    lib.sfgpu_image_warp.argtypes = [C.c_void_p, CP, IP, CP, IP, IP, C.c_int]
    lib.sfgpu_warp_frame_derivs.argtypes = [C.c_void_p, CP, IP, IP, C.c_int, C.c_int, CP, IP, CP, CP, CP, CP, CP]
    lib.sfgpu_compute_dpsis_weight.argtypes = [C.c_void_p, IP, CP, C.c_float, FP, FP, C.c_int]
    lib.sfgpu_compute_smoothness.argtypes = [C.c_void_p, IP, IP, IP, IP, IP, C.c_float, C.c_int, C.c_float,
                                             C.c_float, C.c_int]
    lib.sfgpu_compute_data_and_match.argtypes = [C.c_void_p, IP, IP, IP, IP, IP, IP, IP, IP, CP, CP, C.c_float,
                                                 C.c_float]
    lib.sfgpu_prep_two_frame.argtypes = [C.c_void_p, IP, IP, IP, IP, IP, CP, CP, IP, IP, IP, IP, IP, IP, C.c_float, C.c_float]
    lib.sfgpu_mt_system.argtypes = [C.c_void_p] + [IP] * 7 + [C.POINTER(CP)] + [IP] * 5 + [CP, C.POINTER(MTParams)]
    lib.sfgpu_mt_occ_costs.argtypes = [C.c_void_p, IP, IP, C.POINTER(CP), IP, IP, C.POINTER(MTParams)]
    lib.sfgpu_sub_laplacian.argtypes = [C.c_void_p, IP, IP, IP, IP]
    lib.sfgpu_sor_coupled.argtypes = [C.c_void_p, IP, IP, IP, IP, IP, IP, IP, IP, IP, C.c_int, C.c_float]
    lib.sfgpu_prescale_size.argtypes = [C.c_int, C.c_int, C.c_float, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.sfgpu_prescale.argtypes = [C.c_void_p, CP, CP, C.c_float]
    lib.sfgpu_raw_weighting.argtypes = [C.c_void_p, CP, C.c_int, C.c_int, C.c_float]
    lib.sfgpu_write_flo.argtypes = [C.c_char_p, IP, IP]
    lib.sfgpu_read_flo_size.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.sfgpu_read_flo.argtypes = [C.c_char_p, IP, IP]
    lib.sfgpu_write_occlusion_pbm.argtypes = [C.c_char_p, IP]
    lib.sfgpu_set_device.argtypes = [C.c_int]
    lib.sfgpu_convolve_horiz.argtypes = [C.c_void_p, IP, IP, C.c_int, FP]
    lib.sfgpu_convolve_vert.argtypes = [C.c_void_p, IP, IP, C.c_int, FP]
    lib.sfgpu_color_image_convolve_hv.argtypes = [C.c_void_p, CP, CP, C.c_int, FP, C.c_int, FP]
    lib.sfgpu_get_derivatives.argtypes = [C.c_void_p] + [CP] * 10
    lib.epic_params_default.argtypes = [C.POINTER(EpicParams)]
    lib.epic_params_default.restype = None
    lib.sfgpu_epic.argtypes = [C.c_void_p, IP, IP, CP, C.POINTER(FloatImage), C.POINTER(FloatImage), C.POINTER(EpicParams),
                               C.POINTER(EpicStats)]
    lib.sfgpu_epic_batch.argtypes = [C.c_void_p, C.c_int, C.POINTER(IP), C.POINTER(IP), C.POINTER(CP), C.POINTER(C.POINTER(FloatImage)),
                                     C.POINTER(C.POINTER(FloatImage)), C.POINTER(EpicParams), C.POINTER(EpicStats)]
    lib.sfgpu_rgb_to_lab.argtypes = [C.c_void_p, CP, CP]
    lib.sfgpu_epicflow_sequence.argtypes = [C.c_void_p, C.c_int, C.POINTER(CP), C.POINTER(C.POINTER(FloatImage)),
                                            C.POINTER(C.POINTER(FloatImage)), C.POINTER(EpicParams), VP, C.POINTER(IP), C.POINTER(IP),
                                            C.POINTER(EpicStats)]
    lib.sfgpu_epic_nnfield.argtypes = [C.c_void_p, C.POINTER(C.c_int), FP, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int, C.c_int, FP,
                                       C.c_int, C.c_int, C.POINTER(C.c_int)]
    lib.sfgpu_grid_mincut.argtypes = [C.c_int, C.c_int, FP, FP, C.c_float, C.c_int, C.POINTER(C.c_int)]
    lib.sfgpu_grid_mincut_dev.argtypes = [C.c_void_p, C.c_int, C.c_int, FP, FP, C.c_float, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    if path is None:
        _LIB = lib
    return lib


def epic_params_default():
    p = EpicParams()
    load_library().epic_params_default(C.byref(p))
    return p


def _check(lib, rc, what):
    if rc != 0:
        raise RuntimeError("%s failed (status %d): %s" % (what, rc, lib.sfgpu_last_error().decode()))


def _ip(im):
    return None if im is None else im.ptr()


class Context:
    """An ``sfgpu_ctx``: device + stream + workspace.  Not shareable between host threads."""

    def __init__(self, device=0, stream=None):
        self.lib = load_library()
        h = C.c_void_p()
        _check(self.lib, self.lib.sfgpu_create(int(device), C.c_void_p(stream) if stream else None, C.byref(h)),
               "sfgpu_create")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.sfgpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # --- configuration / timing
    def synchronize(self):
        _check(self.lib, self.lib.sfgpu_synchronize(self.h), "sfgpu_synchronize")

    def set_sor_variant(self, v):
        _check(self.lib, self.lib.sfgpu_set_sor_variant(self.h, int(v)), "sfgpu_set_sor_variant")

    def set_sor_fuse(self, n):
        _check(self.lib, self.lib.sfgpu_set_sor_fuse(self.h, int(n)), "sfgpu_set_sor_fuse")

    def profile_enable(self, on=True):
        _check(self.lib, self.lib.sfgpu_profile_enable(self.h, 1 if on else 0), "sfgpu_profile_enable")

    def profile_reset(self):
        _check(self.lib, self.lib.sfgpu_profile_reset(self.h), "sfgpu_profile_reset")

    def profile_get(self):
        p = Profile()
        _check(self.lib, self.lib.sfgpu_profile_get(self.h, C.byref(p)), "sfgpu_profile_get")
        return p

    # --- two-frame
    def variational(self, wx, wy, im1, im2, params=None):
        _check(self.lib, self.lib.sfgpu_variational(self.h, wx.ptr(), wy.ptr(), im1.ptr(), im2.ptr(),
                                                    C.byref(params) if params is not None else None),
               "sfgpu_variational")

    def variational_dev(self, d_wx, d_wy, d_im1, d_im2, width, height, stride, params=None):
        """Device pointers (ints); asynchronous on the context's stream."""
        _check(self.lib, self.lib.sfgpu_variational_dev(self.h, d_wx, d_wy, d_im1, d_im2, width, height, stride,
                                                        C.byref(params) if params is not None else None),
               "sfgpu_variational_dev")

    def variational_sequence(self, frames, wxs, wys, params=None):
        n = len(wxs)
        assert len(frames) == n + 1 and len(wys) == n
        CP, IP = C.POINTER(color_image_t), C.POINTER(image_t)
        fa = (CP * (n + 1))(*[C.pointer(f.c) for f in frames])
        xa = (IP * n)(*[C.pointer(w.c) for w in wxs])
        ya = (IP * n)(*[C.pointer(w.c) for w in wys])
        _check(self.lib, self.lib.sfgpu_variational_sequence(self.h, n, fa, xa, ya,
                                                             C.byref(params) if params is not None else None),
               "sfgpu_variational_sequence")

    def variational_sequence_int(self, frames, wxs, wys, params=None, continue_from_previous=False):
        """frames: numpy uint8 / uint16 arrays of shape (H, W) or (H, W, 3) (a cv::Mat as the reference's loaders hold
        it before the float conversion, adaptiveFR.cpp:450-464 / slow_flow.cpp:470-477); rows may be strided."""
        import numpy as np
        n = len(wxs)
        assert len(frames) == n + 1 and len(wys) == n
        depth = frames[0].dtype.itemsize * 8
        assert depth in (8, 16) and all(f.dtype == frames[0].dtype for f in frames)
        fa = (FrameInt * (n + 1))()
        for k, f in enumerate(frames):
            ch = 1 if f.ndim == 2 else f.shape[2]
            assert f.strides[1] == ch * f.dtype.itemsize and (f.ndim == 2 or f.strides[2] == f.dtype.itemsize)
            fa[k] = FrameInt(f.shape[1], f.shape[0], ch, f.strides[0], f.ctypes.data)
        IP = C.POINTER(image_t)
        xa = (IP * n)(*[C.pointer(w.c) for w in wxs])
        ya = (IP * n)(*[C.pointer(w.c) for w in wys])
        fn = self.lib.sfgpu_variational_sequence_u8 if depth == 8 else self.lib.sfgpu_variational_sequence_u16
        _check(self.lib, fn(self.h, n, fa, xa, ya, C.byref(params) if params is not None else None,
                            1 if continue_from_previous else 0), "sfgpu_variational_sequence_u%d" % depth)

    # --- EPIC interpolation (epic.cpp:147)
    def epic(self, flowx, flowy, im, matches, edges, params=None):
        """matches: float32 array (n, >= 4) of x1 y1 x2 y2; edges: float32 (H, W) cost map, params.euc is added to it IN
        PLACE like in the reference.  Returns the EpicStats of the call."""
        import numpy as np
        assert matches.dtype == np.float32 and matches.flags.c_contiguous and matches.ndim == 2
        assert edges.dtype == np.float32 and edges.flags.c_contiguous and edges.shape == (im.height, im.width)
        if params is None:
            params = epic_params_default()
        FP = C.POINTER(C.c_float)
        m = FloatImage(matches.ctypes.data_as(FP), matches.shape[1], matches.shape[0])
        e = FloatImage(edges.ctypes.data_as(FP), edges.shape[1], edges.shape[0])
        st = EpicStats()
        _check(self.lib, self.lib.sfgpu_epic(self.h, flowx.ptr(), flowy.ptr(), im.ptr(), C.byref(m), C.byref(e), C.byref(params),
                                             C.byref(st)), "sfgpu_epic")
        return st

    def epic_batch(self, flowsx, flowsy, ims, matches, edges, params=None):
        """epic() on n images of one geometry in one call (sfgpu_epic_batch): item k gets exactly what
        ``epic(flowsx[k], flowsy[k], ims[k], matches[k], edges[k], params)`` gives it.  Same input checks as ``epic``;
        params.euc is added IN PLACE to every edges[k].  Returns the list of the items' EpicStats."""
        import numpy as np
        n = len(flowsx)
        assert len(flowsy) == n and len(ims) == n and len(matches) == n and len(edges) == n
        for im, m, e in zip(ims, matches, edges):
            assert m.dtype == np.float32 and m.flags.c_contiguous and m.ndim == 2
            assert e.dtype == np.float32 and e.flags.c_contiguous and e.shape == (im.height, im.width)
        if params is None:
            params = epic_params_default()
        FP, IP, CP, FIP = C.POINTER(C.c_float), C.POINTER(image_t), C.POINTER(color_image_t), C.POINTER(FloatImage)
        ms = [FloatImage(m.ctypes.data_as(FP), m.shape[1], m.shape[0]) for m in matches]
        es = [FloatImage(e.ctypes.data_as(FP), e.shape[1], e.shape[0]) for e in edges]
        st = (EpicStats * max(n, 1))()
        _check(self.lib, self.lib.sfgpu_epic_batch(self.h, n, (IP * n)(*[C.pointer(f.c) for f in flowsx]),
                                                   (IP * n)(*[C.pointer(f.c) for f in flowsy]), (CP * n)(*[C.pointer(i.c) for i in ims]),
                                                   (FIP * n)(*[C.pointer(m) for m in ms]), (FIP * n)(*[C.pointer(e) for e in es]),
                                                   C.byref(params), st), "sfgpu_epic_batch")
        return list(st[:n])

    def rgb_to_lab(self, src):
        """rgb_to_lab (image.c:694) of a ColorImage in [0, 255] -> a new ColorImage (whole stride rows converted)."""
        dst = ColorImage(src.width, src.height)
        _check(self.lib, self.lib.sfgpu_rgb_to_lab(self.h, dst.ptr(), src.ptr()), "sfgpu_rgb_to_lab")
        return dst

    def epicflow_sequence(self, frames, matches, edges, wxs, wys, epic_params=None, flow_params=None):
        """The EpicFlow two-step over n consecutive pairs of one geometry (sfgpu_epicflow_sequence): pair k writes exactly
        what ``epic(wxs[k], wys[k], rgb_to_lab(frames[k]), matches[k], edges[k], epic_params)`` followed by
        ``variational(wxs[k], wys[k], frames[k], frames[k + 1], flow_params)`` would.  frames: n + 1 RGB ColorImages;
        epic_params.euc is added IN PLACE to every edges[k].  Returns the list of the pairs' EpicStats."""
        import numpy as np
        n = len(wxs)
        assert len(frames) == n + 1 and len(wys) == n and len(matches) == n and len(edges) == n
        for m, e in zip(matches, edges):
            assert m.dtype == np.float32 and m.flags.c_contiguous and m.ndim == 2
            assert e.dtype == np.float32 and e.flags.c_contiguous and e.shape == (frames[0].height, frames[0].width)
        if epic_params is None:
            epic_params = epic_params_default()
        FP, IP, CP, FIP = C.POINTER(C.c_float), C.POINTER(image_t), C.POINTER(color_image_t), C.POINTER(FloatImage)
        ms = [FloatImage(m.ctypes.data_as(FP), m.shape[1], m.shape[0]) for m in matches]
        es = [FloatImage(e.ctypes.data_as(FP), e.shape[1], e.shape[0]) for e in edges]
        st = (EpicStats * max(n, 1))()
        _check(self.lib, self.lib.sfgpu_epicflow_sequence(
            self.h, n, (CP * (n + 1))(*[C.pointer(f.c) for f in frames]), (FIP * max(n, 1))(*[C.pointer(m) for m in ms]),
            (FIP * max(n, 1))(*[C.pointer(e) for e in es]), C.byref(epic_params),
            C.byref(flow_params) if flow_params is not None else None, (IP * max(n, 1))(*[C.pointer(w.c) for w in wxs]),
            (IP * max(n, 1))(*[C.pointer(w.c) for w in wys]), st), "sfgpu_epicflow_sequence")
        return list(st[:n])

    def epic_nnfield(self, seeds, nn, cost):
        """seeds: int32 (ns, 2) x y; cost: float32 (H, W).  -> (labels (H, W), best (ns, nn), dist (ns, nn), sweeps)."""
        import numpy as np
        h, w = cost.shape
        ns = seeds.shape[0]
        labels, best, dist = np.zeros((h, w), np.int32), np.zeros((ns, nn), np.int32), np.zeros((ns, nn), np.float32)
        sweeps = C.c_int()
        IPi, FP = C.POINTER(C.c_int), C.POINTER(C.c_float)
        _check(self.lib, self.lib.sfgpu_epic_nnfield(self.h, best.ctypes.data_as(IPi), dist.ctypes.data_as(FP), labels.ctypes.data_as(IPi),
                                                     np.ascontiguousarray(seeds, np.int32).ctypes.data_as(IPi), ns, nn,
                                                     np.ascontiguousarray(cost, np.float32).ctypes.data_as(FP), w, h, C.byref(sweeps)),
               "sfgpu_epic_nnfield")
        return labels, best, dist, sweeps.value

    # --- multi-frame
    def normalize(self, seq, params):
        CP = C.POINTER(color_image_t)
        arr = (CP * len(seq))(*[C.pointer(f.c) for f in seq])
        _check(self.lib, self.lib.sfgpu_normalize(self.h, arr, len(seq), C.byref(params)), "sfgpu_normalize")

    def variational_mt(self, wx, wy, im, params, channel_w=None, occlusions=None):
        CP = C.POINTER(color_image_t)
        arr = (CP * len(im))(*[C.pointer(f.c) for f in im])
        out = (C.c_float * 2)()
        _check(self.lib, self.lib.sfgpu_variational_mt(self.h, wx.ptr(), wy.ptr(), arr, C.byref(params),
                                                       _ip(channel_w), _ip(occlusions), out),
               "sfgpu_variational_mt")
        return float(out[0]), float(out[1])

    def mt_frame_cache(self, max_frames):
        """Device-side cache of level-0 frames keyed by their host buffers (sfgpu_mt_frame_cache): for callers that solve
        many windows over one immutable sequence.  0 disables."""
        _check(self.lib, self.lib.sfgpu_mt_frame_cache(self.h, int(max_frames)), "sfgpu_mt_frame_cache")

    # --- input side of a window (slow_flow.cpp:538-542, 596-600)
    def prescale(self, src, scale):
        """GaussianBlur + resize by `scale` of a float colour image -> new ColorImage."""
        w, h = C.c_int(), C.c_int()
        _check(self.lib, self.lib.sfgpu_prescale_size(src.width, src.height, scale, C.byref(w), C.byref(h)),
               "sfgpu_prescale_size")
        dst = ColorImage(w.value, h.value)
        _check(self.lib, self.lib.sfgpu_prescale(self.h, dst.ptr(), src.ptr(), scale), "sfgpu_prescale")
        return dst

    def raw_weighting(self, weights, red_x, red_y, weight):
        _check(self.lib, self.lib.sfgpu_raw_weighting(self.h, weights.ptr(), int(red_x), int(red_y), weight),
               "sfgpu_raw_weighting")

    def mt_stats(self):
        s = MTStats()
        _check(self.lib, self.lib.sfgpu_get_mt_stats(self.h, C.byref(s)), "sfgpu_get_mt_stats")
        return s

    # --- operator twins (variational_aux.h:12-29, solver.h:11)
    def image_warp(self, dst, mask, src, wx, wy, factor=1):
        _check(self.lib, self.lib.sfgpu_image_warp(self.h, dst.ptr(), _ip(mask), src.ptr(), wx.ptr(), wy.ptr(),
                                                   int(factor)), "sfgpu_image_warp")

    def warp_frame_derivs(self, src, wx, wy, factor=1, variant=0):
        """warped frame, mask, [Ix, Iy, Ixx, Ixy, Iyy] of the warped frame (the multi-frame path's per-frame pass)"""
        w, h = src.width, src.height
        warped, mask = ColorImage(w, h), Image(w, h)
        outs = [ColorImage(w, h) for _ in range(5)]
        _check(self.lib, self.lib.sfgpu_warp_frame_derivs(self.h, src.ptr(), wx.ptr(), wy.ptr(), int(factor), int(variant),
                                                           warped.ptr(), mask.ptr(), *[o.ptr() for o in outs]),
               "sfgpu_warp_frame_derivs")
        return warped, mask, outs

    def compute_dpsis_weight(self, dst, im, coef=5.0, avg=None, std=None, hbit=0):
        a = (C.c_float * 3)(*avg) if avg is not None else None
        s = (C.c_float * 3)(*std) if std is not None else None
        _check(self.lib, self.lib.sfgpu_compute_dpsis_weight(self.h, dst.ptr(), im.ptr(), coef, a, s, int(hbit)),
               "sfgpu_compute_dpsis_weight")

    def compute_smoothness(self, dst_h, dst_v, uu, vv, w, alpha_factor, robust_reg=-1, eps=0.001, trunc=0.5, mode=1):
        _check(self.lib, self.lib.sfgpu_compute_smoothness(self.h, dst_h.ptr(), dst_v.ptr(), uu.ptr(), vv.ptr(),
                                                           w.ptr(), alpha_factor, int(robust_reg), eps, trunc,
                                                           int(mode)), "sfgpu_compute_smoothness")

    def compute_data_and_match(self, a11, a12, a22, b1, b2, mask, du, dv, im1, im2w, hd, hg):
        _check(self.lib, self.lib.sfgpu_compute_data_and_match(self.h, a11.ptr(), a12.ptr(), a22.ptr(), b1.ptr(),
                                                               b2.ptr(), mask.ptr(), du.ptr(), dv.ptr(), im1.ptr(),
                                                               im2w.ptr(), hd, hg), "sfgpu_compute_data_and_match")

    def prep_two_frame(self, a11, a12, a22, b1, b2, im1, im2, wx, wy, du, dv, ph, pv, hd, hg):
        _check(self.lib, self.lib.sfgpu_prep_two_frame(self.h, a11.ptr(), a12.ptr(), a22.ptr(), b1.ptr(), b2.ptr(), im1.ptr(),
                                                       im2.ptr(), wx.ptr(), wy.ptr(), _ip(du), _ip(dv), ph.ptr(), pv.ptr(), hd, hg),
               "sfgpu_prep_two_frame")

    def mt_system(self, im, wx, wy, params, occ, du=None, dv=None, channel_w=None):
        """One linearisation of the multi-frame solver on one level's frames -> [a11, a12, a22, b1, b2] (blocks inverted)
        and [psi_h, psi_v], whole planes (sfgpu_mt_system)."""
        w, h = wx.width, wx.height
        outs = [Image(w, h) for _ in range(7)]
        arr = (C.POINTER(color_image_t) * len(im))(*[C.pointer(f.c) for f in im])
        _check(self.lib, self.lib.sfgpu_mt_system(self.h, *[o.ptr() for o in outs], arr, wx.ptr(), wy.ptr(), _ip(du), _ip(dv),
                                                  occ.ptr(), _ip(channel_w), C.byref(params)), "sfgpu_mt_system")
        return outs[:5], outs[5:]

    def mt_occ_costs(self, im, wx, wy, params):
        """Occlusion data costs (d0, d1) of one level's frames at (wx, wy) (sfgpu_mt_occ_costs)."""
        d0, d1 = Image(wx.width, wx.height), Image(wx.width, wx.height)
        arr = (C.POINTER(color_image_t) * len(im))(*[C.pointer(f.c) for f in im])
        _check(self.lib, self.lib.sfgpu_mt_occ_costs(self.h, d0.ptr(), d1.ptr(), arr, wx.ptr(), wy.ptr(), C.byref(params)),
               "sfgpu_mt_occ_costs")
        return d0, d1

    def convolve(self, dst, src, coeffs, vertical=False):
        """convolve_horiz / convolve_vert (image.c:400-645) with 3 or 5 taps."""
        arr = (C.c_float * len(coeffs))(*coeffs)
        fn = self.lib.sfgpu_convolve_vert if vertical else self.lib.sfgpu_convolve_horiz
        _check(self.lib, fn(self.h, dst.ptr(), src.ptr(), (len(coeffs) - 1) // 2, arr), "sfgpu_convolve")

    def color_image_convolve_hv(self, dst, src, horiz=None, vert=None):
        ha = (C.c_float * len(horiz))(*horiz) if horiz is not None else None
        va = (C.c_float * len(vert))(*vert) if vert is not None else None
        _check(self.lib, self.lib.sfgpu_color_image_convolve_hv(self.h, dst.ptr(), src.ptr(),
                                                                (len(horiz) - 1) // 2 if horiz is not None else 0, ha,
                                                                (len(vert) - 1) // 2 if vert is not None else 0, va),
               "sfgpu_color_image_convolve_hv")

    def get_derivatives(self, im1, im2):
        """-> [dx, dy, dt, dxx, dxy, dyy, dxt, dyt] (variational_aux.c:55-78)."""
        outs = [ColorImage(im1.width, im1.height) for _ in range(8)]
        _check(self.lib, self.lib.sfgpu_get_derivatives(self.h, im1.ptr(), im2.ptr(), *[o.ptr() for o in outs]),
               "sfgpu_get_derivatives")
        return outs

    def sub_laplacian(self, dst, src, wh, wv):
        _check(self.lib, self.lib.sfgpu_sub_laplacian(self.h, dst.ptr(), src.ptr(), wh.ptr(), wv.ptr()),
               "sfgpu_sub_laplacian")

    def sor_coupled(self, du, dv, a11, a12, a22, b1, b2, ph, pv, iterations, omega):
        _check(self.lib, self.lib.sfgpu_sor_coupled(self.h, du.ptr(), dv.ptr(), a11.ptr(), a12.ptr(), a22.ptr(),
                                                    b1.ptr(), b2.ptr(), ph.ptr(), pv.ptr(), int(iterations), omega),
               "sfgpu_sor_coupled")


def variational(wx, wy, im1, im2, params=None):
    """Legacy drop-in entry (variational.c:101): refines wx, wy in place; aborts the process on error
    exactly like the reference (fprintf + exit(1))."""
    lib = load_library()
    lib.variational(wx.ptr(), wy.ptr(), im1.ptr(), im2.ptr(), C.byref(params) if params is not None else None)


class Variational_MT:
    """Shape of the reference class (variational_mt.h:23-71) over ``sfgpu_variational_mt``."""

    def __init__(self, ctx=None):
        self.ctx = ctx or Context()
        self.one_direction = False
        self._channel_w = None
        self._occlusions = None

    def setChannelWeights(self, weights):
        self._channel_w = weights

    def getOcclusions(self):
        return self._occlusions

    def variational(self, wx, wy, im, params):
        p = params
        if self.one_direction and not p.one_direction:
            p = MTParams.from_buffer_copy(bytes(params))
            p.one_direction = 1
        self._occlusions = Image(wx.width, wx.height)
        return self.ctx.variational_mt(wx, wy, im, p, self._channel_w, self._occlusions)


def write_flo(path, wx, wy):
    """writeFlowFile (epic_flow_extended/io.c:78-96)."""
    lib = load_library()
    _check(lib, lib.sfgpu_write_flo(str(path).encode(), wx.ptr(), wy.ptr()), "sfgpu_write_flo")


def read_flo(path):
    """readFlowFile (epic_flow_extended/io.c:50-75) -> (wx, wy)."""
    lib = load_library()
    w, h = C.c_int(), C.c_int()
    _check(lib, lib.sfgpu_read_flo_size(str(path).encode(), C.byref(w), C.byref(h)), "sfgpu_read_flo_size")
    wx, wy = Image(w.value, h.value), Image(w.value, h.value)
    _check(lib, lib.sfgpu_read_flo(str(path).encode(), wx.ptr(), wy.ptr()), "sfgpu_read_flo")
    return wx, wy


def write_occlusion_pbm(path, occ):
    """Occlusion labels as slow_flow.cpp:893-905 stores them."""
    lib = load_library()
    _check(lib, lib.sfgpu_write_occlusion_pbm(str(path).encode(), occ.ptr()), "sfgpu_write_occlusion_pbm")
