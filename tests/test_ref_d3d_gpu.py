"""Pin the oracle AND the product against the reference's own D3D extension (3D/dcn, CUDA-only).  What that extension computed,
compiled for sm_100a by oracle/build_ref.py (two-token torch-2 patch, see that file) and run on a B200 by
tests/golden/make_golden_d3d.py, is stored in tests/golden/ref3d_d3d.npz; the inputs are regenerated here from the same seeds.
A stored tensor keeps its shape, its largest magnitude and its values at the positions sample_index picks (all of them for a
small tensor); errors are relative to that largest magnitude."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle.oracle import _triple, out_extent

DEV = "cuda:0"
GOLD = os.path.join(GOLDEN, "ref3d_d3d.npz")
GRAD_NAMES = ("grad_input", "grad_offset", "grad_weight", "grad_bias")

FORWARD_CASES = [   # C, Co, g, dg, k, s, p, d, offset scale
    (8, 8, 1, 1, 3, 1, 1, 1, 1.0),
    (16, 12, 1, 1, 3, 1, 1, 1, 8.0),
    (16, 16, 2, 2, (3, 2, 3), (1, 2, 1), (1, 0, 2), (1, 2, 1), 2.0),
]
BACKWARD_CASES = [(8, 12, (6, 7, 9), 1.5), (32, 32, (8, 8, 8), 0.5), (16, 16, (24, 20, 20), 0.5)]   # C, Co, dims, scale
GROUP_CASES = [(16, 8, 2, 1, (5, 6, 7), 0.7), (16, 16, 1, 2, (6, 5, 7), 1.5), (32, 24, 2, 4, (4, 6, 5), 0.7)]   # + g, dg


def sample_index(n, k):
    """k positions of a flat tensor of n elements, a prime stride apart (modulo n), so no axis of the tensor is favoured;
    all n when n <= k."""
    if n <= k:
        return torch.arange(n)
    assert n % 1000003
    return torch.arange(k, dtype=torch.int64) * 1000003 % n


def forward_inputs(C, Co, g, dg, k, s, p, d, scale):
    torch.manual_seed(0)
    B, D, H, W = 2, 6, 7, 9
    kd, kh, kw = _triple(k); sd, sh, sw = _triple(s); pd, ph, pw = _triple(p); dd, dh, dw = _triple(d)
    Do, Ho, Wo = out_extent(D, pd, dd, kd, sd), out_extent(H, ph, dh, kh, sh), out_extent(W, pw, dw, kw, sw)
    x = torch.randn(B, C, D, H, W); w = torch.randn(Co, C // g, kd, kh, kw) * 0.2; b = torch.randn(Co)
    off = torch.randn(B, dg * 3 * kd * kh * kw, Do, Ho, Wo) * scale
    return x, w, b, off


def c3_inputs():
    """BASELINE config 3: (2,64,32,64,64), k=3 -- the largest shape class the reference's int32 indexing survives."""
    torch.manual_seed(1)
    B, C, D, H, W = 2, 64, 32, 64, 64
    x = torch.randn(B, C, D, H, W, device=DEV); w = torch.randn(C, C, 3, 3, 3, device=DEV) * 0.05
    b = torch.randn(C, device=DEV); off = torch.randn(B, 81, D, H, W, device=DEV)
    return x, w, b, off


def backward_inputs(C, Co, g, dg, dims, scale, seed):
    torch.manual_seed(seed)
    B = 2
    D, H, W = dims
    x = torch.randn(B, C, D, H, W); w = torch.randn(Co, C // g, 3, 3, 3) * 0.2; b = torch.randn(Co)
    off = torch.randn(B, dg * 81, D, H, W) * scale
    gout = torch.randn(B, Co, D, H, W)
    return x, w, b, off, gout


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def check(gold, key, got, tol, what=""):
    """max |got - ref| over the stored positions, over max |ref| of the whole reference tensor, below tol; and the largest
    magnitude of the whole of `got` within the same bound."""
    shape = tuple(int(n) for n in gold[key + ".shape"])
    assert tuple(got.shape) == shape, (what, key, tuple(got.shape), shape)
    ref = torch.from_numpy(gold[key + ".values"])
    absmax = float(gold[key + ".absmax"])
    got = got.detach().float().cpu().reshape(-1)
    err = (got[sample_index(got.numel(), ref.numel())] - ref).abs().max().item() / absmax
    assert err < tol, (what, key, err)
    assert abs(got.abs().max().item() - absmax) / absmax < tol, (what, key, "largest magnitude")


@pytest.mark.parametrize("C,Co,g,dg,k,s,p,d,scale", FORWARD_CASES)
def test_oracle_matches_compiled_reference(gold, oracle, C, Co, g, dg, k, s, p, d, scale):
    x, w, b, off = forward_inputs(C, Co, g, dg, k, s, p, d, scale)
    ora = oracle.deform_conv3d(x, off, w, b, s, p, d, g, dg)
    check(gold, f"forward{FORWARD_CASES.index((C, Co, g, dg, k, s, p, d, scale))}", ora, 1e-5)


@pytest.mark.gpu
def test_product_matches_compiled_reference_at_c3_shape(gold):
    import deformablelka_b200 as dl
    x, w, b, off = c3_inputs()
    assert torch.equal(x.flatten()[:16].cpu(), torch.from_numpy(gold["c3.x_head"]))   # same input as the reference saw
    for math in ("fp32", "bf16x3"):
        got = dl.ops.deform_conv3d_forward(x, w, b, off, 3, 1, 1, 1, 1, 1, 64, math=math)
        check(gold, "c3", got, 1e-3, math)


@pytest.mark.gpu
@pytest.mark.parametrize("C,Co,dims,scale", BACKWARD_CASES)
def test_backward_matches_compiled_reference(gold, oracle, C, Co, dims, scale):
    """Row N2 against the reference's own D3D.deform_conv_backward (deform_conv_cuda.cu:128-285) at the block's configuration
    k = 3, stride 1, pad (1,1,1), dilation 1: with equal pads on every axis the reference's pad_h/pad_w index defect
    (deform_im2col_cuda.cuh:448) has no effect, so its four gradients are the exact target; the autograd oracle is checked
    against it on the way (pins the backward oracle to the real reference)."""
    import deformablelka_b200 as dl
    x, w, b, off, gout = backward_inputs(C, Co, 1, 1, dims, scale, seed=2)
    key = f"backward{BACKWARD_CASES.index((C, Co, dims, scale))}"
    if x.numel() < 200000:   # the pure-torch autograd oracle is for small shapes
        xo, wo, bo, oo = (t.clone().requires_grad_() for t in (x, w, b, off))
        oracle.deform_conv3d_autograd(xo, oo, wo, bo).backward(gout)
        for n, o_ in zip(GRAD_NAMES, (xo.grad, oo.grad, wo.grad, bo.grad)):
            check(gold, f"{key}.{n}", o_, 2e-5, "oracle")
    for math in ("fp32", "bf16x3"):
        got = dl.ops.deform_conv3d_backward(x.to(DEV), w.to(DEV), b.to(DEV), off.to(DEV), gout.to(DEV), 3, 1, 1, 1, 1, 1, 64, math=math)
        for n, g_ in zip(GRAD_NAMES, got):
            check(gold, f"{key}.{n}", g_, 1e-3, math)


@pytest.mark.gpu
@pytest.mark.parametrize("C,Co,g,dg,dims,scale", GROUP_CASES)
def test_backward_groups_match_compiled_reference(gold, oracle, C, Co, g, dg, dims, scale):
    """group / deformable_group != 1 in the backward (deform_conv_cuda.cu:160-166, 204-270), against the reference's own compiled
    D3D.deform_conv_backward; same equal-pad argument as above.  The grouped autograd oracle is pinned on the way."""
    import deformablelka_b200 as dl
    x, w, b, off, gout = backward_inputs(C, Co, g, dg, dims, scale, seed=3)
    key = f"groups{GROUP_CASES.index((C, Co, g, dg, dims, scale))}"
    xo, wo, bo, oo = (t.clone().requires_grad_() for t in (x, w, b, off))
    oracle.deform_conv3d_autograd(xo, oo, wo, bo, (1, 1, 1), (1, 1, 1), (1, 1, 1), g, dg).backward(gout)
    for n, o_ in zip(GRAD_NAMES, (xo.grad, oo.grad, wo.grad, bo.grad)):
        check(gold, f"{key}.{n}", o_, 2e-5, "oracle")
    for math in ("fp32", "bf16x3"):
        got = dl.ops.deform_conv3d_backward(x.to(DEV), w.to(DEV), b.to(DEV), off.to(DEV), gout.to(DEV), 3, 1, 1, 1, g, dg, 64, math=math)
        for n, g_ in zip(GRAD_NAMES, got):
            check(gold, f"{key}.{n}", g_, 1e-3, math)
