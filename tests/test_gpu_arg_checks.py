"""Every entry that takes image_t / color_image_t host buffers refuses a malformed image argument before it touches anything
(the container contract of include/slowflow_gpu.h, checked by arg_geom / arg_is in slowflow_b200/csrc/sf_context.cu).

For each entry and each of its image arguments, that one argument gets one fault: null data, width + 1, height + 1, stride
ceil4(width) + 4, or (colour images) c3 = c2.  The call must return SFGPU_ERR_ARG (2), sfgpu_last_error() must name the entry
and the argument, and no caller buffer may change: image planes with the guard region behind them, edge maps, matches,
integer frames, stats and parameters.  Each image struct points at the start of a buffer far larger than any copy an entry
could derive from a faulted geometry, and every stride is a multiple of 4, so a missing check fails an assertion here
instead of reading or writing memory it should not."""
import ctypes as C

import numpy as np
import pytest

import mt_helpers
from slowflow_b200 import synth
from slowflow_b200.api import EpicStats, FloatImage, FrameInt, epic_params_default
from slowflow_b200.image import _aligned, ceil4, color_image_t, image_t

pytestmark = pytest.mark.gpu

W, H = 32, 24  # a width that is a multiple of 4: width + 1 needs another stride
PW, PH = 16, 12  # what sfgpu_prescale_size reports for W x H at scale 0.5
CAP = 4 * 3 * (ceil4(W) + 8) * (H + 8)  # floats behind every image struct
SENTINEL = np.float32(-12345.5)
FP, IP, CP = C.POINTER(C.c_float), C.POINTER(image_t), C.POINTER(color_image_t)
FAULTS = ("null", "width", "height", "stride", "c3")


class Buf:
    """An image_t ('i') or color_image_t ('c') of w x h at the start of CAP floats: the planes hold values in [0, 1), the
    rest is a guard region of SENTINEL."""

    def __init__(self, kind, w, h, seed):
        self.kind, self.w, self.h = kind, w, h
        self.a = _aligned(CAP)
        self.a[:] = SENTINEL
        n = (3 if kind == "c" else 1) * ceil4(w) * h
        self.a[:n] = np.random.RandomState(seed).rand(n)
        self.orig = self.a.copy()

    def struct(self, fault=None):
        w, h, s = self.w, self.h, ceil4(self.w)
        P, base = s * h, self.a.ctypes.data  # the planes stay where the buffer has them, whatever the fault
        w, h, s = w + (fault == "width"), h + (fault == "height"), s + 4 * (fault == "stride")
        at = lambda off: C.cast(base + 4 * off, FP)
        data = None if fault == "null" else at(0)
        if self.kind == "i":
            return image_t(w, h, s, data)
        return color_image_t(w, h, s, data, at(P), at(P if fault == "c3" else 2 * P))

    def unchanged(self):
        return np.array_equal(self.a.view(np.uint32), self.orig.view(np.uint32))


def arr(ptr_type, ptrs):
    return (ptr_type * len(ptrs))(*ptrs)


def float_images(arrays):
    return [FloatImage(a.ctypes.data_as(FP), a.shape[1], a.shape[0]) for a in arrays]


def epic_extras(n):
    """matches, edge maps (numpy, in place), their float_image structs, EPIC parameters and stats of n items"""
    cases = [synth.epic_case(W, H, 30, seed=70 + k) for k in range(n)]
    x = dict(matches=[np.ascontiguousarray(m) for _, m, _ in cases], edges=[np.ascontiguousarray(e) for _, _, e in cases],
             params=epic_params_default(), stats=(EpicStats * n)())
    x["fm"], x["fe"] = float_images(x["matches"]), float_images(x["edges"])
    return x


def int_frames(depth):
    t = np.uint8 if depth == 8 else np.uint16
    raw = [np.random.RandomState(90 + f).randint(0, 256, (H, W, 3)).astype(t) for f in range(3)]
    return dict(raw=raw, frames=(FrameInt * 3)(*[FrameInt(W, H, 3, W * 3 * raw[0].itemsize, r.ctypes.data) for r in raw]))


class Entry:
    """images: (name, kind) of the entry's image arguments, the one that gives the call's geometry first; `items` numbers
    the arrays in `itemized` ("pair" / "item"); call(lib, handle, I, X) -> status, I: name -> struct pointer, X: the other
    caller buffers."""

    def __init__(self, name, images, call, extras=dict, items=None, itemized=(), geometry=None):
        self.name, self.images, self.call, self.extras = name, images, call, extras
        self.items, self.itemized, self.geometry = items, itemized, geometry or {}

    def expected(self, arg):
        base, _, k = arg.partition("[")
        if base in self.itemized:
            return "%s %s: %s: " % (self.items, k[:-1], base)
        return ": %s: " % arg


def images(spec):
    """'wx:i wy:i im1:c' -> [('wx', 'i'), ('wy', 'i'), ('im1', 'c')]"""
    return [tuple(a.split(":")) for a in spec.split()]


def seq(name, n, kind):
    return " ".join("%s[%d]:%s" % (name, k, kind) for k in range(n))


MT = mt_helpers.params(S=2)
COEF = (C.c_float * 5)(1 / 12, -8 / 12, 0, 8 / 12, -1 / 12)
DERIVS = "dx dy dt dxx dxy dyy dxt dyt"

ENTRIES = [
    Entry("sfgpu_variational", images("wx:i wy:i im1:c im2:c"),
          lambda L, h, I, X: L.sfgpu_variational(h, I["wx"], I["wy"], I["im1"], I["im2"], None)),
    Entry("sfgpu_image_warp", images("src:c dst:c mask:i wx:i wy:i"),
          lambda L, h, I, X: L.sfgpu_image_warp(h, I["dst"], I["mask"], I["src"], I["wx"], I["wy"], 1)),
    Entry("sfgpu_warp_frame_derivs", images("src:c wx:i wy:i mask:i warped:c dx:c dy:c dxx:c dxy:c dyy:c"),
          lambda L, h, I, X: L.sfgpu_warp_frame_derivs(h, I["src"], I["wx"], I["wy"], 1, 0, I["warped"], I["mask"], I["dx"], I["dy"],
                                                       I["dxx"], I["dxy"], I["dyy"])),
    Entry("sfgpu_convolve_horiz", images("src:i dst:i"), lambda L, h, I, X: L.sfgpu_convolve_horiz(h, I["dst"], I["src"], 2, COEF)),
    Entry("sfgpu_convolve_vert", images("src:i dst:i"), lambda L, h, I, X: L.sfgpu_convolve_vert(h, I["dst"], I["src"], 2, COEF)),
    Entry("sfgpu_color_image_convolve_hv", images("src:c dst:c"),
          lambda L, h, I, X: L.sfgpu_color_image_convolve_hv(h, I["dst"], I["src"], 2, COEF, 2, COEF)),
    Entry("sfgpu_get_derivatives", images("im1:c im2:c " + " ".join(d + ":c" for d in DERIVS.split())),
          lambda L, h, I, X: L.sfgpu_get_derivatives(h, I["im1"], I["im2"], *[I[d] for d in DERIVS.split()])),
    Entry("sfgpu_compute_dpsis_weight", images("im:c dst:i"),
          lambda L, h, I, X: L.sfgpu_compute_dpsis_weight(h, I["dst"], I["im"], 5.0, None, None, 0)),
    Entry("sfgpu_compute_smoothness", images("uu:i vv:i dpsis_weight:i dst_horiz:i dst_vert:i"),
          lambda L, h, I, X: L.sfgpu_compute_smoothness(h, I["dst_horiz"], I["dst_vert"], I["uu"], I["vv"], I["dpsis_weight"], 0.5,
                                                        -1, 0.0, 0.0, 1)),
    Entry("sfgpu_compute_data_and_match", images("im1:c im2w:c mask:i du:i dv:i a11:i a12:i a22:i b1:i b2:i"),
          lambda L, h, I, X: L.sfgpu_compute_data_and_match(h, I["a11"], I["a12"], I["a22"], I["b1"], I["b2"], I["mask"], I["du"], I["dv"],
                                                            I["im1"], I["im2w"], 0.0, 0.1)),
    Entry("sfgpu_prep_two_frame", images("wx:i wy:i im1:c im2:c du:i dv:i dpsis_horiz:i dpsis_vert:i a11:i a12:i a22:i b1:i b2:i"),
          lambda L, h, I, X: L.sfgpu_prep_two_frame(h, I["a11"], I["a12"], I["a22"], I["b1"], I["b2"], I["im1"], I["im2"], I["wx"], I["wy"],
                                                    I["du"], I["dv"], I["dpsis_horiz"], I["dpsis_vert"], 0.0, 0.1)),
    Entry("sfgpu_sub_laplacian", images("src:i dst:i weight_horiz:i weight_vert:i"),
          lambda L, h, I, X: L.sfgpu_sub_laplacian(h, I["dst"], I["src"], I["weight_horiz"], I["weight_vert"])),
    Entry("sfgpu_sor_coupled", images("du:i dv:i a11:i a12:i a22:i b1:i b2:i dpsis_horiz:i dpsis_vert:i"),
          lambda L, h, I, X: L.sfgpu_sor_coupled(h, I["du"], I["dv"], I["a11"], I["a12"], I["a22"], I["b1"], I["b2"], I["dpsis_horiz"],
                                                 I["dpsis_vert"], 5, 1.9)),
    Entry("sfgpu_variational_mt", images("wx:i wy:i channel_w:c occlusions_out:i " + seq("im", 3, "c")),
          lambda L, h, I, X: L.sfgpu_variational_mt(h, I["wx"], I["wy"], arr(CP, [I["im[%d]" % f] for f in range(3)]), X["params"],
                                                    I["channel_w"], I["occlusions_out"], X["avg"]),
          extras=lambda: dict(params=mt_helpers.clone_params(MT), avg=(C.c_float * 2)(7.0, 7.0))),
    Entry("sfgpu_normalize", images(seq("seq", 3, "c")),
          lambda L, h, I, X: L.sfgpu_normalize(h, arr(CP, [I["seq[%d]" % f] for f in range(3)]), 3, X["params"]),
          extras=lambda: dict(params=mt_helpers.clone_params(MT))),
    Entry("sfgpu_prescale", images("src:c dst:c"), lambda L, h, I, X: L.sfgpu_prescale(h, I["dst"], I["src"], 0.5),
          geometry={"dst": (PW, PH)}),
    Entry("sfgpu_raw_weighting", images("weights:c"), lambda L, h, I, X: L.sfgpu_raw_weighting(h, I["weights"], 0, 0, 1.0)),
    Entry("sfgpu_rgb_to_lab", images("src:c dst:c"), lambda L, h, I, X: L.sfgpu_rgb_to_lab(h, I["dst"], I["src"])),
    Entry("sfgpu_epic", images("im:c flowx:i flowy:i"),
          lambda L, h, I, X: L.sfgpu_epic(h, I["flowx"], I["flowy"], I["im"], C.pointer(X["fm"][0]), C.pointer(X["fe"][0]), X["params"], X["stats"]),
          extras=lambda: epic_extras(1)),
    Entry("sfgpu_epic_batch", images(" ".join([seq("im", 2, "c"), seq("flowx", 2, "i"), seq("flowy", 2, "i")])),
          lambda L, h, I, X: L.sfgpu_epic_batch(h, 2, *[arr(IP, [I["%s[%d]" % (a, k)] for k in range(2)]) for a in ("flowx", "flowy")],
                                                arr(CP, [I["im[0]"], I["im[1]"]]), arr(C.POINTER(FloatImage), [C.pointer(m) for m in X["fm"]]),
                                                arr(C.POINTER(FloatImage), [C.pointer(m) for m in X["fe"]]), X["params"], X["stats"]),
          extras=lambda: epic_extras(2), items="item", itemized=("im", "flowx", "flowy")),
    Entry("sfgpu_variational_sequence", images(" ".join([seq("wx", 2, "i"), seq("wy", 2, "i"), seq("frames", 3, "c")])),
          lambda L, h, I, X: L.sfgpu_variational_sequence(h, 2, arr(CP, [I["frames[%d]" % f] for f in range(3)]),
                                                          *[arr(IP, [I["%s[%d]" % (a, k)] for k in range(2)]) for a in ("wx", "wy")], None),
          items="pair", itemized=("wx", "wy")),
    Entry("sfgpu_epicflow_sequence", images(" ".join([seq("frames", 3, "c"), seq("wx", 2, "i"), seq("wy", 2, "i")])),
          lambda L, h, I, X: L.sfgpu_epicflow_sequence(h, 2, arr(CP, [I["frames[%d]" % f] for f in range(3)]),
                                                       arr(C.POINTER(FloatImage), [C.pointer(m) for m in X["fm"]]), arr(C.POINTER(FloatImage), [C.pointer(m) for m in X["fe"]]), X["params"],
                                                       None, *[arr(IP, [I["%s[%d]" % (a, k)] for k in range(2)]) for a in ("wx", "wy")],
                                                       X["stats"]),
          extras=lambda: epic_extras(2), items="pair", itemized=("wx", "wy")),
] + [
    Entry("sfgpu_variational_sequence_u%d" % d, images(" ".join([seq("wx", 2, "i"), seq("wy", 2, "i")])),
          lambda L, h, I, X, d=d: getattr(L, "sfgpu_variational_sequence_u%d" % d)(
              h, 2, X["frames"], *[arr(IP, [I["%s[%d]" % (a, k)] for k in range(2)]) for a in ("wx", "wy")], None, 0),
          extras=lambda d=d: int_frames(d), items="pair", itemized=("wx", "wy"))
    for d in (8, 16)
]
BY_NAME = {e.name: e for e in ENTRIES}

# The first image argument an entry reads gives the call's geometry.  An image_t one height + 1 is a consistent image of
# another size; the next argument is then the one reported as of a different geometry.
SOURCE = {e.name: e.images[0][0] for e in ENTRIES}
CASES = [(e.name, a, f) for e in ENTRIES for a, kind in e.images for f in FAULTS
         if (f != "c3" or kind == "c") and not (a == "occlusions_out" and f == "null")]  # (no labels wanted: skipped)


def snapshot(x):
    """bytes of every caller buffer in an entry's extras"""
    out = []
    for v in x.values():
        for item in (v if isinstance(v, list) else [v]):
            out.append(item.tobytes() if isinstance(item, np.ndarray) else bytes(item))
    return out


@pytest.mark.parametrize("entry,arg,fault", CASES)
def test_malformed_image_argument_is_refused_untouched(ctx, entry, arg, fault):
    e = BY_NAME[entry]
    bufs = {a: Buf(kind, *e.geometry.get(a, (W, H)), seed=k) for k, (a, kind) in enumerate(e.images)}
    structs = {a: b.struct(fault if a == arg else None) for a, b in bufs.items()}
    x = e.extras()
    before = snapshot(x)
    rc = e.call(ctx.lib, ctx.h, {a: C.pointer(s) for a, s in structs.items()}, x)
    msg = ctx.lib.sfgpu_last_error().decode()
    assert rc == 2, (rc, msg)
    assert msg.startswith(e.name + ": "), msg
    if arg == SOURCE[entry] and fault == "height" and e.images[0][1] == "i":
        assert "different geometry" in msg, msg
    else:
        assert e.expected(arg) in msg, msg
    assert all(b.unchanged() for b in bufs.values()), [a for a, b in bufs.items() if not b.unchanged()]
    assert snapshot(x) == before
