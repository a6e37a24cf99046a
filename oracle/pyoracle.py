"""ctypes loader for the CPU checkers under oracle/.  TEST INFRASTRUCTURE ONLY.

Importers allowed: tests/, __graft_entry__.smoke(), bench.py's cpu_baseline / --impl reference
legs.  The product package ``slowflow_b200`` never imports this module.

  Oracle()      -> oracle/libsf_oracle.so      (our C restatement, `make -C oracle oracle`)
  Reference()   -> oracle/_ref/libsf_ref.so    (the reference's own sources compiled in place,
                                                `make -C oracle ref`; prebuilt where /root/reference
                                                is absent)
"""
import ctypes as C
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(_HERE))
from slowflow_b200.image import image_t, color_image_t  # noqa: E402  (shared struct layout only)
from slowflow_b200.params import VariationalParams, MTParams  # noqa: E402

ORACLE_SO = os.path.join(_HERE, "libsf_oracle.so")
REF_SO = os.path.join(_HERE, "_ref", "libsf_ref.so")
SOR_LEX, SOR_REDBLACK = 0, 1


def build(ref=True):
    """(Re)build the checkers; the reference build is skipped where /root/reference is absent."""
    subprocess.check_call(["make", "-s", "-C", _HERE, "oracle"])
    if ref:
        subprocess.check_call(["make", "-s", "-C", _HERE, "ref"])


def have_reference():
    return os.path.exists(REF_SO)


IP, CP, VP = C.POINTER(image_t), C.POINTER(color_image_t), C.POINTER(VariationalParams)


class Oracle:
    """Our restatement (sf_oracle.c / sf_oracle_mt.c)."""

    def __init__(self):
        if not os.path.exists(ORACLE_SO):
            build(ref=False)
        L = self.lib = C.CDLL(ORACLE_SO, mode=os.RTLD_LOCAL)
        L.sfo_variational.argtypes = [IP, IP, CP, CP, VP, C.c_int]
        L.sfo_image_warp.argtypes = [CP, IP, CP, IP, IP, C.c_int]
        L.sfo_get_derivatives.argtypes = [CP] * 10
        L.sfo_compute_smoothness.argtypes = [IP, IP, IP, IP, IP, C.c_float]
        L.sfo_sub_laplacian.argtypes = [IP, IP, IP, IP]
        L.sfo_compute_dpsis_weight.argtypes = [CP, C.c_float]
        L.sfo_compute_dpsis_weight.restype = IP
        L.sfo_image_delete.argtypes = [IP]
        L.sfo_compute_data_and_match.argtypes = [IP] * 8 + [CP] * 8 + [C.c_float, C.c_float]
        L.sfo_sor_coupled.argtypes = [IP] * 9 + [C.c_int, C.c_float, C.c_int]
        L.sfo_sor_coupled_readable.argtypes = [IP] * 9 + [C.c_int, C.c_float]
        if hasattr(L, "sfo_variational_mt"):
            L.sfo_variational_mt.argtypes = [IP, IP, C.POINTER(CP), C.POINTER(MTParams), CP, IP,
                                             C.POINTER(C.c_float), C.c_int, C.POINTER(C.c_int)]
            L.sfo_normalize.argtypes = [C.POINTER(CP), C.c_int, C.POINTER(MTParams)]
            L.sfo_mt_smoothness.argtypes = [IP] * 5 + [C.c_float, C.c_int, C.c_int, C.c_float, C.c_float]
            L.sfo_mt_dpsis_weight.argtypes = [IP, CP, C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int]
            L.sfo_mt_system.argtypes = [IP] * 7 + [C.POINTER(CP)] + [IP] * 5 + [CP, C.POINTER(MTParams)]
            L.sfo_mt_occ_costs.argtypes = [IP, IP, C.POINTER(CP), IP, IP, C.POINTER(MTParams)]

    def variational(self, wx, wy, im1, im2, params=None, sor_mode=SOR_LEX):
        self.lib.sfo_variational(wx.ptr(), wy.ptr(), im1.ptr(), im2.ptr(),
                                 C.byref(params) if params is not None else None, sor_mode)


class Reference:
    """The reference's own objects (+ glue).  Two-frame: unmodified variational.c & co."""

    def __init__(self):
        if not os.path.exists(REF_SO):
            raise RuntimeError("oracle/_ref/libsf_ref.so missing (needs /root/reference to build)")
        L = self.lib = C.CDLL(REF_SO, mode=os.RTLD_LOCAL)
        L.variational.argtypes = [IP, IP, CP, CP, VP]
        L.variational.restype = None
        L.sf_ref_set_sor_mode.argtypes = [C.c_int]
        L.image_warp.argtypes = [CP, IP, CP, IP, IP]
        L.get_derivatives.argtypes = [CP, CP, C.c_void_p] + [CP] * 8
        L.compute_smoothness.argtypes = [IP, IP, IP, IP, IP, C.c_void_p, C.c_float]
        L.sub_laplacian.argtypes = [IP, IP, IP, IP]
        L.compute_dpsis_weight.argtypes = [CP, C.c_float, C.c_void_p]
        L.compute_dpsis_weight.restype = IP
        L.compute_data_and_match.argtypes = [IP] * 8 + [CP] * 8 + [C.c_float, C.c_float]
        L.sor_coupled.argtypes = [IP] * 9 + [C.c_int, C.c_float]
        L.sor_coupled_slow_but_readable.argtypes = [IP] * 9 + [C.c_int, C.c_float]
        L.convolution_new.argtypes = [C.c_int, C.POINTER(C.c_float), C.c_int]
        L.convolution_new.restype = C.c_void_p
        L.image_delete.argtypes = [IP]
        self.deriv = L.convolution_new(2, (C.c_float * 3)(0.0, -8.0 / 12.0, 1.0 / 12.0), 0)
        self.deriv_flow = L.convolution_new(1, (C.c_float * 2)(0.0, -0.5), 0)
        if hasattr(L, "sf_ref_variational_mt"):
            L.sf_ref_variational_mt.argtypes = [IP, IP, C.POINTER(CP), C.POINTER(MTParams), CP, IP,
                                                C.POINTER(C.c_float), C.c_int, C.POINTER(C.c_int)]
            L.sf_ref_normalize.argtypes = [C.POINTER(CP), C.c_int, C.POINTER(MTParams)]

    def variational(self, wx, wy, im1, im2, params=None, sor_mode=SOR_LEX):
        self.lib.sf_ref_set_sor_mode(sor_mode)
        try:
            self.lib.variational(wx.ptr(), wy.ptr(), im1.ptr(), im2.ptr(),
                                 C.byref(params) if params is not None else None)
        finally:
            self.lib.sf_ref_set_sor_mode(SOR_LEX)
