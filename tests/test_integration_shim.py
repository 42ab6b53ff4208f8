"""INTEGRATION.md section 1 as a tested file: deformablelka_b200/compat/D3D.py is imported under the reference's module name
``D3D`` and driven with the reference's own calling sequence (3D/dcn/functions/deform_conv_func.py:15-56, restated in
``_RefDeformConvFunction`` below -- argument order, the kernel-size / stride / padding / dilation unpacking and the order of the
four returned gradients are what that file does with the compiled extension)."""
import importlib
import importlib.util
import inspect
import json
import os
import sys

import pytest
import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable
from torch.nn.modules.utils import _triple

from conftest import GOLDEN, ROOT

SHIM = os.path.join(ROOT, "deformablelka_b200", "compat", "D3D.py")


@pytest.fixture(scope="module")
def D3D():
    spec = importlib.util.spec_from_file_location("D3D", SHIM)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_shim_exports_the_reference_signatures(D3D):
    fwd = list(inspect.signature(D3D.deform_conv_forward).parameters)
    bwd = list(inspect.signature(D3D.deform_conv_backward).parameters)
    geom = ["kd", "kh", "kw", "sd", "sh", "sw", "pd", "ph", "pw", "dd", "dh", "dw", "group", "deformable_group", "im2col_step"]
    assert fwd == ["input", "weight", "bias", "offset"] + geom            # deform_conv.h:10-28
    assert bwd == ["input", "weight", "bias", "offset", "grad_output"] + geom   # deform_conv.h:49-68
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        D3D.deform_conv_forward(torch.randn(1, 4, 3, 3, 3), torch.randn(4, 4, 3, 3, 3), torch.zeros(4), torch.zeros(1, 81, 3, 3, 3),
                                3, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 64)


def test_reference_function_source_calls_match_the_shim(D3D):
    """The reference's deform_conv_func.py as recorded in tests/golden/ref3d_deform_conv_func.json (make_golden_shim.py): with
    the shim as ``D3D`` every import it makes resolves, and its Function's forward / backward call exactly the two shim entry
    points, each with as many positional arguments as the shim function takes."""
    rec = json.load(open(os.path.join(GOLDEN, "ref3d_deform_conv_func.json")))
    assert ["D3D", None] in rec["imports"]
    sys.modules["D3D"] = D3D
    try:
        for module, name in rec["imports"]:
            mod = importlib.import_module(module)
            assert name is None or hasattr(mod, name), (module, name)
    finally:
        sys.modules.pop("D3D", None)
    assert [(c["caller"], c["function"]) for c in rec["d3d_calls"]] == [
        ("DeformConvFunction.forward", "deform_conv_forward"), ("DeformConvFunction.backward", "deform_conv_backward")]
    for c in rec["d3d_calls"]:
        assert len(inspect.signature(getattr(D3D, c["function"])).parameters) == c["positional_args"], c


def _make_ref_function(D3D):
    class _RefDeformConvFunction(Function):   # calling sequence of 3D/dcn/functions/deform_conv_func.py:15-56
        @staticmethod
        def forward(ctx, input, offset, weight, bias, stride, padding, dilation, group, deformable_groups, im2col_step):
            ctx.stride, ctx.padding, ctx.dilation = _triple(stride), _triple(padding), _triple(dilation)
            ctx.kernel_size = _triple(weight.shape[2:5])
            ctx.group, ctx.deformable_groups, ctx.im2col_step = group, deformable_groups, im2col_step
            out = D3D.deform_conv_forward(input, weight, bias, offset, *ctx.kernel_size, *ctx.stride, *ctx.padding, *ctx.dilation,
                                          ctx.group, ctx.deformable_groups, ctx.im2col_step)
            ctx.save_for_backward(input, offset, weight, bias)
            return out

        @staticmethod
        @once_differentiable
        def backward(ctx, grad_output):
            input, offset, weight, bias = ctx.saved_tensors
            gi, go, gw, gb = D3D.deform_conv_backward(input, weight, bias, offset, grad_output, *ctx.kernel_size, *ctx.stride,
                                                      *ctx.padding, *ctx.dilation, ctx.group, ctx.deformable_groups, ctx.im2col_step)
            return gi, go, gw, gb, None, None, None, None, None, None
    return _RefDeformConvFunction


@pytest.mark.gpu
def test_shim_forward_backward_through_the_reference_calling_sequence(D3D, oracle):
    torch.manual_seed(0)
    dev = "cuda:0"
    B, C, Co, dims = 2, 16, 16, (5, 6, 7)
    x = torch.randn(B, C, *dims, requires_grad=True)
    w = (torch.randn(Co, C, 3, 3, 3) * 0.2).requires_grad_()
    b = torch.randn(Co, requires_grad=True)
    off = (torch.randn(B, 81, *dims) * 0.8).requires_grad_()
    gout = torch.randn(B, Co, *dims)
    ref = oracle.deform_conv3d_autograd(x, off, w, b)
    ref.backward(gout)
    F = _make_ref_function(D3D)
    xg, og, wg, bg = (t.detach().to(dev).requires_grad_() for t in (x, off, w, b))
    y = F.apply(xg, og, wg, bg, 1, 1, 1, 1, 1, 64)
    y.backward(gout.to(dev))
    rel = lambda a, r: ((a.detach().cpu() - r).abs().max() / r.abs().max()).item()
    assert rel(y, ref.detach()) < 1e-3
    for got, want in ((xg.grad, x.grad), (og.grad, off.grad), (wg.grad, w.grad), (bg.grad, b.grad)):
        assert rel(got, want) < 1e-3
