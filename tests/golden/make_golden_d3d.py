"""Golden vectors for tests/test_ref_d3d_gpu.py: the reference's own D3D extension (3D/dcn, CUDA-only), compiled for sm_100a by
oracle/build_ref.py into oracle/_ref/, run on the inputs the tests regenerate from their seeds.  Needs a B200 and oracle/_ref/:

    python tests/golden/make_golden_d3d.py [OUT.npz]        (default: tests/golden/ref3d_d3d.npz)

Every tensor is stored as its shape, its largest magnitude and its values at test_ref_d3d_gpu.sample_index positions.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]
import test_ref_d3d_gpu as t  # noqa: E402
from oracle import build_ref  # noqa: E402

SAMPLE = 1024        # stored values per tensor
SAMPLE_C3 = 8192     # the 16.8M-element output of the C3 shape


def put(out, key, ref, k=SAMPLE):
    ref = ref.detach().float().cpu()
    out[key + ".shape"] = np.asarray(ref.shape, dtype=np.int64)
    out[key + ".absmax"] = np.float64(ref.abs().max())
    out[key + ".values"] = ref.reshape(-1)[t.sample_index(ref.numel(), k)].numpy()


def main(path):
    d3d = build_ref.load_d3d()
    assert d3d is not None, "oracle/_ref/D3D*.so not built (python oracle/build_ref.py)"
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = t.DEV
    out = {}
    for i, (C, Co, g, dg, k, s, p, d, scale) in enumerate(t.FORWARD_CASES):
        x, w, b, off = (v.to(dev) for v in t.forward_inputs(C, Co, g, dg, k, s, p, d, scale))
        put(out, f"forward{i}", d3d.deform_conv_forward(x, w, b, off, *t._triple(k), *t._triple(s), *t._triple(p), *t._triple(d),
                                                        g, dg, 64))
    x, w, b, off = t.c3_inputs()
    out["c3.x_head"] = x.flatten()[:16].cpu().numpy()
    put(out, "c3", d3d.deform_conv_forward(x, w, b, off, 3, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 64), SAMPLE_C3)
    del x, off
    cases = [("backward", i, C, Co, 1, 1, dims, scale, 2) for i, (C, Co, dims, scale) in enumerate(t.BACKWARD_CASES)]
    cases += [("groups", i, *case, 3) for i, case in enumerate(t.GROUP_CASES)]
    for prefix, i, C, Co, g, dg, dims, scale, seed in cases:
        x, w, b, off, gout = (v.to(dev) for v in t.backward_inputs(C, Co, g, dg, dims, scale, seed))
        grads = d3d.deform_conv_backward(x, w, b, off, gout, 3, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, g, dg, 64)
        for n, r in zip(t.GRAD_NAMES, grads):
            put(out, f"{prefix}{i}.{n}", r)
    np.savez_compressed(path, **out)
    print(f"wrote {path}: {os.path.getsize(path) / 1e3:.0f} kB, {len(out)} arrays")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "ref3d_d3d.npz"))
