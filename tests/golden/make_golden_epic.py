"""Generates tests/golden/epic_gpu_regression.npz: the outputs of this project's GPU path (sfgpu_epic_nnfield, sfgpu_epic) on
the cases of tests/epic_helpers.py.  These are regression vectors of the GPU code, not outputs of the original project.
Needs a CUDA device.  Regenerate only for an intended change of results.

    python tests/golden/make_golden_epic.py [OUT_DIR]
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from slowflow_b200 import Context, Image  # noqa: E402
import epic_helpers as eh  # noqa: E402


def main(out_dir):
    out = {}
    with Context(0) as ctx:
        for w, h, ns, nn, kind in eh.REGRESSION_NNFIELD:
            t = eh.tag(w, h, ns, nn, kind)
            seeds, cost = eh.nnfield_inputs(w, h, ns, kind)
            labels, best, dist, _ = ctx.epic_nnfield(seeds, nn, cost)
            out["labels_" + t], out["best_" + t], out["dist_" + t] = eh.stored(labels), eh.stored(best), eh.stored(dist)
        for w, h, n, method, filters in eh.REGRESSION_EPIC:
            t = eh.tag(w, h, n, method, filters)
            ci, m, edges, p = eh.epic_inputs(w, h, n, method, filters)
            fx, fy = Image(w, h), Image(w, h)
            st = ctx.epic(fx, fy, ci, m, edges, p)
            out["counts_" + t] = np.array([st.matches_in, st.matches_after_saliency, st.matches_after_consistency], np.int32)
            out["edges_" + t] = eh.stored(edges, eh.FLOW_SAMPLE)
            out["fx_" + t], out["fy_" + t] = eh.stored(fx.array, eh.FLOW_SAMPLE), eh.stored(fy.array, eh.FLOW_SAMPLE)
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, os.path.basename(eh.REGRESSION_FILE))
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.dirname(eh.REGRESSION_FILE))
