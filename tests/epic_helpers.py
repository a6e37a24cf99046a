"""Seeded inputs of the EPIC tests (test_gpu_epic.py) and the cases and sampling of the stored regression vectors
(tests/golden/epic_gpu_regression.npz, written by tests/golden/make_golden_epic.py)."""
import os

import numpy as np

from slowflow_b200 import ColorImage, synth
from slowflow_b200.api import epic_params_default

REGRESSION_FILE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "epic_gpu_regression.npz")
# every distance-transform and interpolation case of the reference comparisons in test_gpu_epic.py
REGRESSION_NNFIELD = [(97, 61, 40, 10, "texture"), (200, 150, 300, 26, "texture"), (64, 64, 64, 26, "flat"),
                      (333, 211, 900, 100, "texture"), (1024, 436, 5000, 100, "texture"), (130, 33, 50, 50, "ridges"),
                      (31, 7, 12, 5, "texture"), (100, 5, 9, 4, "texture"), (96, 32, 30, 10, "texture"), (97, 33, 30, 10, "ridges"),
                      (70, 50, 25, 8, "zero")]
REGRESSION_EPIC = [(320, 200, 800, "LA", True), (320, 200, 800, "NW", True), (1024, 436, 5000, "LA", True), (501, 333, 2500, "LA", True),
                   (160, 120, 37, "LA", False)]
WHOLE = 32768      # label maps and neighbour tables up to this many entries are stored whole, larger ones on a sample of it
SAMPLE = 4096      # entries of that sample
FLOW_SAMPLE = 1024  # pixels at which the dense flows and the edge map are stored


def unique_seeds(w, h, n, seed):
    r = np.random.RandomState(seed)
    p = r.permutation(w * h)[:n]
    return np.stack([p % w, p // w], axis=1).astype(np.int32)


def nnfield_inputs(w, h, ns, kind):
    """-> (seeds (ns, 2), cost (H, W)) of one distance-transform case."""
    _, _, cost = synth.epic_case(w, h, 10)
    if kind == "flat":
        cost = np.full((h, w), 0.25, np.float32)  # constant cost: ties everywhere
    elif kind == "ridges":
        cost = cost + (np.arange(w)[None, :] % 17 == 0) * 5.0  # expensive ridges: many sweeps until nothing changes
        cost = cost.astype(np.float32)
    cost = np.ascontiguousarray(cost + np.float32(0.001))
    if kind == "zero":
        cost = np.zeros((h, w), np.float32)
    return unique_seeds(w, h, ns, w * 7 + ns), cost


def epic_inputs(w, h, n, method, filters=True):
    """-> (image, matches, edges, params) of one interpolation case; filters=False: saliency_th = pref_nn = 0 and no outliers."""
    im, m, edges = synth.epic_case(w, h, n) if filters else synth.epic_case(w, h, n, outliers=0.0)
    p = epic_params_default()
    p.method = method.encode()
    if not filters:
        p.saliency_th, p.pref_nn = 0.0, 0
    return ColorImage.from_array(im), m, edges, p


def tag(*case):
    return "_".join(str(c) for c in case)


def stored(a, k=None):
    """The entries of array `a` that the regression file keeps: all of them up to WHOLE, else a fixed seeded sample of SAMPLE
    (k: that many instead, always sampled)."""
    a = np.asarray(a).reshape(-1)
    if k is None and a.size <= WHOLE:
        return a
    k = min(k or SAMPLE, a.size)
    return a[np.sort(np.random.RandomState(a.size).choice(a.size, k, replace=False))]
