#!/usr/bin/env python
"""oracle/make_golden_ref_op.py -- run the reference's own CUDA op (oracle/_ref, built by build_ref.py) and store its outputs.

TEST INFRASTRUCTURE.  Needs a GPU and oracle/_ref/MultiScaleDeformableAttention.so, which only exists where the reference
sources were at build time; its product, tests/golden/msda_ref_op.npz, lets tests/test_msda_gpu.py compare our MSDA
operator with the reference op on any machine with a GPU.

  python oracle/make_golden_ref_op.py [OUT_DIR]        (default: tests/golden)

Inputs are regenerated from seeds by oracle.synth (the same calls as the tests), so only outputs are stored:
  fwd.<dtype>.<Lq>.<border>.sha256   SHA-256 of every output value (signed zeros folded to +0), for the bit-exact check;
  fwd.<dtype>.<Lq>.<border>.sample   the output at fwd.<Lq>.idx (a seeded sample of flat indices), for the error message;
  bwd.<grad>.sample / .absmax / .idx a seeded sample of each gradient and its max |.| over the whole tensor (the rel_err
                                     denominator).  The backward accumulates with atomics, so it is compared to a tolerance.
"""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import synth  # noqa: E402

S = sum(h * w for h, w in synth.DANCETRACK_SHAPES)
# (the cases of test_forward_bit_exact_vs_reference_cuda_op and test_backward_full_encoder_size_vs_c_oracle_and_reference_op)
FWD_CASES = [(dtype, Lq, border) for dtype in (torch.float32, torch.float64) for Lq, border in ((400, False), (S, True))]
FWD_SAMPLE, BWD_SAMPLE = 1024, 4096


def fwd_inputs(dtype, Lq, border):
    return synth.msda_inputs(synth.DANCETRACK_SHAPES, B=2, H=8, D=32, K=4, Lq=Lq, seed=50, border=border, dtype=dtype)


def bwd_inputs():
    t = synth.msda_inputs(synth.DANCETRACK_SHAPES, B=1, H=8, D=32, K=4, Lq=S, seed=43, border=True)
    go = torch.randn(1, S, 256, generator=torch.Generator().manual_seed(44))
    return t, go


def fwd_key(dtype, Lq, border):
    return f"fwd.{str(dtype).split('.')[-1]}.{Lq}.{int(border)}"


def bits_sha256(a):
    """SHA-256 of the values of `a` (numpy); -0.0 and +0.0 hash alike, as torch.equal treats them."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256((a + a.dtype.type(0)).tobytes()).hexdigest()


def sample_index(n, k, seed):
    return np.sort(np.random.default_rng(seed).choice(n, size=min(k, n), replace=False)).astype(np.int32)


def main(out_dir):
    sys.path.insert(0, os.path.join(HERE, "_ref"))
    import MultiScaleDeformableAttention as MSDA
    dev = torch.device("cuda")
    out = {}
    for dtype, Lq, border in FWD_CASES:
        t = tuple(x.to(dev) for x in fwd_inputs(dtype, Lq, border))
        y = MSDA.ms_deform_attn_forward(*t, 64).cpu().numpy()
        idx_key = f"fwd.{Lq}.idx"
        if idx_key not in out:
            out[idx_key] = sample_index(y.size, FWD_SAMPLE, seed=Lq)
        k = fwd_key(dtype, Lq, border)
        out[k + ".sha256"] = np.asarray(bits_sha256(y))
        out[k + ".sample"] = y.reshape(-1)[out[idx_key]]
    t, go = bwd_inputs()
    grads = MSDA.ms_deform_attn_backward(*(x.to(dev) for x in t), go.to(dev), 64)
    for seed, (name, g) in enumerate(zip(("grad_value", "grad_loc", "grad_attn"), grads)):
        g = g.cpu().numpy()
        idx = sample_index(g.size, BWD_SAMPLE, seed=100 + seed)
        out[f"bwd.{name}.idx"] = idx
        out[f"bwd.{name}.sample"] = g.reshape(-1)[idx].astype(np.float32)
        out[f"bwd.{name}.absmax"] = np.asarray(np.abs(g).max(), dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "msda_ref_op.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes,", len(out), "arrays")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden"))
