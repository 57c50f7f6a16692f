"""GPU parity against the reference's OWN CUDA kernels.  Those kernels (compiled for sm_100a by oracle/Makefile `ref`) were
run on a B200 on exactly these inputs by tests/golden/make_golden_refcuda.py; what they computed is stored in
tests/golden/refcuda_<case>.npz as a fixed sample of every output (full tensors of the C2 cases are tens of MB)."""
import numpy as np
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu


CASES = {
    "c1_enc": (1, 8, 32, [(60, 80), (30, 40), (15, 20), (8, 10)], 4, None),
    "c2_dec_n2": (2, 8, 32, [(100, 167), (50, 84), (25, 42), (13, 21)], 4, 300),
    "d36_l8": (1, 8, 36, [(17, 30), (9, 15), (5, 8), (3, 4)] * 2, 4, 311),
    "ref_test_shape": (2, 2, 4, [(8, 8), (4, 4), (2, 2)], 2, 3),
}
OUTPUTS = ("out", "grad_value", "grad_loc", "grad_attn")
INPUTS = ("value", "loc", "attn", "grad_out")


def sample_index(numel, k=2048):
    """k distinct flat indices spread over the tensor (i * p mod numel with p a prime above every numel here), or all."""
    if numel <= k:
        return np.arange(numel)
    return (np.arange(k, dtype=np.int64) * 2147483647 + 12345) % numel


def sample(t, k=2048):
    flat = t.detach().reshape(-1).cpu()
    return flat[torch.from_numpy(sample_index(flat.numel(), k))].numpy()


def make_inputs(name, dev):
    N, M, D, hw, P, Lq = CASES[name]
    g = torch.Generator().manual_seed(len(name))
    shapes = torch.as_tensor(hw, dtype=torch.long)
    S = int((shapes[:, 0] * shapes[:, 1]).sum())
    Lq = S if Lq is None else Lq
    L = len(hw)
    value = torch.randn(N, S, M, D, generator=g).to(dev)
    loc = (torch.rand(N, Lq, M, L, P, 2, generator=g) * 1.2 - 0.1).to(dev)
    attn = torch.softmax(torch.randn(N, Lq, M, L * P, generator=g), -1).view(N, Lq, M, L, P).to(dev)
    gout = torch.randn(N, Lq, M * D, generator=g).to(dev)
    return dict(value=value, shapes=shapes.to(dev), loc=loc, attn=attn, grad_out=gout)


@pytest.mark.parametrize("name", sorted(CASES))
def test_matches_reference_cuda_kernels(cuda_device, name):
    from trackformer_b200 import ext
    msda = ext.load()
    gold = load_golden(name, prefix="refcuda_")
    x = make_inputs(name, cuda_device)
    for k in INPUTS:                                   # the inputs the reference kernels saw (same seeded CPU generator)
        np.testing.assert_array_equal(sample(x[k], 256), gold["in_" + k], err_msg=f"input {k} differs from the recorded one")
    value, shapes, loc, attn, gout = (x[k] for k in ("value", "shapes", "loc", "attn", "grad_out"))
    out = msda.ms_deform_attn_forward(value, shapes, loc, attn, 64)
    gv, gl, ga = msda.ms_deform_attn_backward(value, shapes, loc, attn, gout, 64)
    got = dict(zip(OUTPUTS, (out, gv, gl, ga)))
    for k in OUTPUTS:
        assert tuple(got[k].shape) == tuple(gold["shape_" + k]), k
    scale = max(1.0, float(gold["grad_value_absmax"]))
    np.testing.assert_allclose(sample(out), gold["out"], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(sample(gv), gold["grad_value"], rtol=1e-4, atol=1e-4 * scale)
    np.testing.assert_allclose(sample(ga), gold["grad_attn"], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(sample(gl), gold["grad_loc"], rtol=5e-4, atol=5e-3)
