"""Stored reference outputs for test_gpu_production_shapes.py::test_k100_config2_vs_unmodified_reference_on_this_gpu: K=100
at BASELINE config 2 (n=1000, 500+500, hidden_dim 800, --scaling, 16 instances) computed the reference's way in stock
PyTorch fp32 on the GPU (helpers.k100_reference_record; the file's `source` says whether the reference's own modules or the
oracle's restatement of them produced it).  The test compares against this file when baseline/_ref is absent.

    python tests/golden/make_k100_config2_golden.py        # on a GPU; writes tests/golden/k100_config2.npz
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from helpers import K100_SHAPE, K100_ROWS, k100_reference_record      # noqa: E402


def main(device="cuda:0", path=os.path.join(HERE, "k100_config2.npz")):
    rec, source = k100_reference_record(device)
    meta = [K100_SHAPE[k] for k in ("B", "n", "mi", "me", "h", "K", "seed")]
    np.savez_compressed(path, source=np.array(source), meta=np.array(meta), rows=np.array(K100_ROWS),
                        **{k: v.numpy() for k, v in rec.items()})
    print(path, os.path.getsize(path), "bytes |", source)


if __name__ == "__main__":
    main()
