"""Regenerates tests/golden/ref_nn.npz: the indices the REFERENCE'S OWN nearest-neighbour kernel
(lib/utils/extend_utils/src/nearest_neighborhood.cu, compiled verbatim into oracle/_ref/libpvnet_refnn.so by
oracle/metrics.mk, target `refnn`) returns on the inputs of tests/metrics_cases.py.

Needs a CUDA device and oracle/_ref only:

    python tests/golden/make_golden_nn.py [OUT_DIR]        (default: tests/golden)

For every case of nn_cases(): `<name>_in`, the digest (tests.helpers.digest) of the rebuilt inputs, and
`<name>_idx`, the reference's int32 indices.  For the large cases (LARGE): the input digest and the digest of
the indices.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_nn  # noqa: E402
from tests.helpers import digest  # noqa: E402
from tests.metrics_cases import large_nn_case, nn_cases  # noqa: E402

# name -> (seed, b, pn1, pn2, dim): many queries per image, and few queries against a large reference set
LARGE = {"large3": (7, 4, 8192, 8192, 3), "large2": (8, 4, 8192, 8192, 2), "few_queries3": (9, 1, 200003, 96, 3)}


def main():
    if not ref_nn.available():
        raise SystemExit(f"{ref_nn.LIB_PATH} and a CUDA device are needed")
    dst = sys.argv[1] if len(sys.argv) > 1 else HERE
    os.makedirs(dst, exist_ok=True)
    out = {}
    for name, (ref, que, excl) in nn_cases().items():
        out[f"{name}_in"] = np.array(digest(np.concatenate([ref.ravel(), que.ravel()])))
        out[f"{name}_idx"] = ref_nn.find_nearest_point_idx_batched(ref, que, excl)
    for name, case in LARGE.items():
        ref, que = large_nn_case(*case)
        out[f"{name}_in"] = np.array(digest(np.concatenate([ref.ravel(), que.ravel()])))
        out[f"{name}_idx"] = np.array(digest(ref_nn.find_nearest_point_idx_batched(ref, que)))
    path = os.path.join(dst, "ref_nn.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
