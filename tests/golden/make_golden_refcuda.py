#!/usr/bin/env python
"""Records the reference's own CUDA kernels on the cases of tests/test_refcuda_gpu.py.

Needs a CUDA device and oracle/_ref/libmsda_refcuda.so (``make -f oracle/Makefile ref``, where the reference
sources are):  ``python tests/golden/make_golden_refcuda.py [OUT_DIR]``  (default: tests/golden).

For each case it stores refcuda_<case>.npz: a fixed sample of every output (forward output and the three gradients),
each output's full shape, the full-tensor max |grad_value| the test scales its tolerance with, and a sample of every
input so that the test can tell when its seeded generator no longer yields the inputs recorded here.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from oracle import refcuda  # noqa: E402
from test_refcuda_gpu import CASES, INPUTS, OUTPUTS, make_inputs, sample  # noqa: E402


def main(out_dir):
    assert torch.cuda.is_available() and refcuda.available(), "needs a CUDA device and oracle/_ref/libmsda_refcuda.so"
    dev = torch.device("cuda:0")
    os.makedirs(out_dir, exist_ok=True)
    for name in sorted(CASES):
        x = make_inputs(name, dev)
        args = (x["value"], x["shapes"], x["loc"], x["attn"])
        got = dict(zip(OUTPUTS, (refcuda.forward(*args), *refcuda.backward(*args, x["grad_out"]))))
        torch.cuda.synchronize()
        rec = {k: sample(v) for k, v in got.items()}
        rec.update({"shape_" + k: np.asarray(v.shape, dtype=np.int64) for k, v in got.items()})
        rec.update({"in_" + k: sample(x[k], 256) for k in INPUTS})
        rec["grad_value_absmax"] = np.float32(got["grad_value"].abs().max().item())
        path = os.path.join(out_dir, f"refcuda_{name}.npz")
        np.savez_compressed(path, **rec)
        print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else HERE)
