"""GPU parity tests of the MSDA operator through the C ABI (run on the B200 box: `pytest -m gpu`).

Checker hierarchy
  1. oracle/msda.py   (plain-C restatement, fma=True)        -> fp32 forward must be BIT-IDENTICAL
  2. tests/golden/msda_core.npz (the reference's own ms_deform_attn_core_pytorch, produced in the authoring
     container)                                               -> models/ops/test.py tolerances and tighter
  3. tests/golden/msda_ref_op.npz (what the reference CUDA op itself computed on the DanceTrack shapes, stored by
     oracle/make_golden_ref_op.py)                            -> forward BIT-IDENTICAL (SHA-256 of every output value),
                                                                 backward to tolerance on a seeded sample
  4. size-independent properties at the full encoder size (linearity in value, partition of unity).
"""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_err
from oracle import make_golden_ref_op as ref_op
from oracle import msda as omsda
from oracle import synth

pytestmark = pytest.mark.gpu

G = np.load(os.path.join(GOLDEN, "msda_core.npz"))
R = np.load(os.path.join(GOLDEN, "msda_ref_op.npz"))
CASES = sorted({k.split(".")[0] for k in G.files})
DEV = "cuda"


def _mod():
    import memotr_b200
    return memotr_b200


def _inputs(name, dtype):
    B, H, D, K, Lq, seed, border = (int(x) for x in G[name + ".meta"])
    shapes = [tuple(int(v) for v in r) for r in G[name + ".shapes"]]
    return synth.msda_inputs(shapes, B=B, H=H, D=D, K=K, Lq=Lq, seed=seed, border=bool(border), dtype=dtype)


def _fwd(t):
    m = _mod()
    return m.ms_deform_attn_forward(*(x.to(DEV) for x in t), 64)


# ------------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("name", CASES)
def test_forward_fp32_bit_exact_vs_c_oracle(name):
    t = _inputs(name, torch.float32)
    got = _fwd(t).cpu().numpy()
    want = omsda.forward(*(x.numpy() for x in t), fma=True)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), rel_err(got, want)


@pytest.mark.parametrize("name", CASES)
def test_forward_vs_reference_golden(name):
    t32, t64 = _inputs(name, torch.float32), _inputs(name, torch.float64)
    got32, got64 = _fwd(t32).cpu().numpy(), _fwd(t64).cpu().numpy()
    assert np.allclose(got64, G[name + ".fwd64"], rtol=1e-5, atol=1e-8)        # models/ops/test.py:40
    assert np.allclose(got32, G[name + ".fwd32"], rtol=1e-2, atol=1e-3)        # models/ops/test.py:56
    assert rel_err(got64, G[name + ".fwd64"]) < 1e-12
    assert rel_err(got32, G[name + ".fwd64"]) < 1e-4                           # north-star fp32 tolerance


@pytest.mark.parametrize("name", ["tiny_d32", "cfg1", "cfg1_border"])
def test_forward_bf16(name):
    t = _inputs(name, torch.float32)
    tb = tuple(x.to(torch.bfloat16) if x.is_floating_point() else x for x in t)
    got = _fwd(tb).float().cpu().numpy()
    # checker: the fp32 oracle fed the same bf16-rounded inputs (isolates kernel error from input rounding)
    want = omsda.forward(*(x.float().numpy() if x.is_floating_point() else x.numpy() for x in tb), fma=True)
    assert rel_err(got, want) < 1e-2                                            # north-star bf16 tolerance


@pytest.mark.parametrize("K", [1, 2, 3, 4, 8, 16])
@pytest.mark.parametrize("shapes", [synth.BDD_SHAPES, synth.BDD_SHAPES_L5])
def test_forward_point_and_level_sweep(K, shapes):
    """BASELINE.json config #5 geometry (K in {4,8,16}, L in {4,5}) plus odd K; Lq kept small for the CPU oracle."""
    t = synth.msda_inputs(shapes, B=1, H=8, D=32, K=K, Lq=64, seed=20 + K, border=True)
    got = _fwd(t).cpu().numpy()
    want = omsda.forward(*(x.numpy() for x in t), fma=True)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("D", [1, 2, 30, 64, 71])
def test_forward_generic_channel_counts(D):
    t = synth.msda_inputs(((6, 4), (3, 2)), B=2, H=2, D=D, K=2, Lq=5, seed=30 + D, border=True)
    got = _fwd(t).cpu().numpy()
    want = omsda.forward(*(x.numpy() for x in t), fma=True)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_forward_full_encoder_size_bit_exact():
    """Lq = S = 22323 queries x 8 heads x 16 points: the encoder-shaped call of the DanceTrack config."""
    S = sum(h * w for h, w in synth.DANCETRACK_SHAPES)
    t = synth.msda_inputs(synth.DANCETRACK_SHAPES, B=1, H=8, D=32, K=4, Lq=S, seed=41, border=True)
    got = _fwd(t).cpu().numpy()
    want = omsda.forward(*(x.numpy() for x in t), fma=True)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_forward_bit_exact_vs_reference_cuda_op():
    for dtype, Lq, border in ref_op.FWD_CASES:
        t = tuple(x.to(DEV) for x in ref_op.fwd_inputs(dtype, Lq, border))
        ours = _mod().ms_deform_attn_forward(*t, 64).cpu().numpy()
        k = ref_op.fwd_key(dtype, Lq, border)
        got, want = ours.reshape(-1)[R[f"fwd.{Lq}.idx"]], R[k + ".sample"]
        assert np.array_equal(got, want), (k, np.abs(got - want).max())
        assert ref_op.bits_sha256(ours) == str(R[k + ".sha256"]), k


def test_forward_properties_full_size():
    S = sum(h * w for h, w in synth.DANCETRACK_SHAPES)
    value, shp, lsi, loc, attn = (x.to(DEV) for x in synth.msda_inputs(synth.DANCETRACK_SHAPES, Lq=S, seed=42))
    f = _mod().ms_deform_attn_forward
    # linearity in value
    v2 = torch.rand_like(value)
    lhs = f(value + v2, shp, lsi, loc, attn, 64)
    rhs = f(value, shp, lsi, loc, attn, 64) + f(v2, shp, lsi, loc, attn, 64)
    assert rel_err(lhs.cpu().numpy(), rhs.cpu().numpy()) < 1e-5
    # partition of unity: constant value map + interior samples + weights summing to 1 => the constant
    loc_in = loc * 0.8 + 0.1
    ones = torch.full_like(value, 3.0)
    out = f(ones, shp, lsi, loc_in, attn, 64)
    assert torch.allclose(out, torch.full_like(out, 3.0), rtol=1e-5, atol=1e-5)
    # all samples outside the open interval (-1, size): exact zeros
    out = f(value, shp, lsi, loc + 3.0, attn, 64)
    assert torch.count_nonzero(out) == 0


def test_forward_empty_and_errors():
    m = _mod()
    value, shp, lsi, loc, attn = (x.to(DEV) for x in synth.msda_inputs(((6, 4), (3, 2)), H=2, D=32, K=2, Lq=3))
    assert m.ms_deform_attn_forward(value, shp, lsi, loc[:, :0], attn[:, :0], 64).shape == (1, 0, 64)
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        m.ms_deform_attn_forward(value.cpu(), shp.cpu(), lsi.cpu(), loc.cpu(), attn.cpu(), 64)
    with pytest.raises(RuntimeError, match="contiguous"):
        m.ms_deform_attn_forward(value.transpose(2, 3), shp, lsi, loc, attn, 64)
    with pytest.raises(RuntimeError):
        m.ms_deform_attn_forward(value, shp, lsi, loc, attn[:, :, :1], 64)
    with pytest.raises(RuntimeError):
        m.ms_deform_attn_forward(value.half(), shp, lsi, loc.half(), attn.half(), 64)


# ------------------------------------------------------------------------------------------------ backward
def _bwd(t, go):
    return [g.cpu().numpy() for g in _mod().ms_deform_attn_backward(*(x.to(DEV) for x in t), go.to(DEV), 64)]


@pytest.mark.parametrize("name", CASES)
def test_backward_fp64_vs_reference_autograd(name):
    t = _inputs(name, torch.float64)
    gv, gl, ga = _bwd(t, torch.from_numpy(G[name + ".grad_out"]))
    assert rel_err(gl, G[name + ".grad_loc"]) < 1e-10
    assert rel_err(ga, G[name + ".grad_attn"]) < 1e-10
    if name + ".grad_value" in G.files:
        assert rel_err(gv, G[name + ".grad_value"]) < 1e-10
    else:
        r = torch.randn(32, generator=torch.Generator().manual_seed(12), dtype=torch.float64).numpy()
        assert rel_err(gv.sum(-1), G[name + ".grad_value_sumD"]) < 1e-5
        assert rel_err((gv * r).sum(-1), G[name + ".grad_value_dotD"]) < 1e-5


@pytest.mark.parametrize("name", CASES)
def test_backward_fp32_vs_c_oracle(name):
    t = _inputs(name, torch.float32)
    go = torch.from_numpy(G[name + ".grad_out"]).float()
    gv, gl, ga = _bwd(t, go)
    wv, wl, wa = omsda.backward(*(x.numpy() for x in t), go.numpy())
    for got, want in ((gv, wv), (gl, wl), (ga, wa)):
        assert rel_err(got, want) < 1e-5


def test_backward_full_encoder_size_vs_c_oracle_and_reference_op():
    t, go = ref_op.bwd_inputs()
    gv, gl, ga = _bwd(t, go)
    wv, wl, wa = omsda.backward(*(x.numpy() for x in t), go.numpy())
    assert rel_err(gv, wv) < 1e-5 and rel_err(gl, wl) < 1e-5 and rel_err(ga, wa) < 1e-5
    for name, g in (("grad_value", gv), ("grad_loc", gl), ("grad_attn", ga)):
        got = g.reshape(-1)[R[f"bwd.{name}.idx"]]
        err = np.abs(got - R[f"bwd.{name}.sample"]).max() / R[f"bwd.{name}.absmax"]
        assert err < 1e-5, (name, err)


@pytest.mark.parametrize("channels", [30, 32, 64, 71, 1025, 2048, 3096])      # the reference list, models/ops/test.py:85-86
def test_gradcheck_like_reference(channels):
    """models/ops/test.py:63-78 -- torch.autograd.gradcheck in fp64 through MSDeformAttnFunction."""
    from torch.autograd import gradcheck
    value, shp, lsi, loc, attn = synth.msda_inputs(((6, 4), (3, 2)), B=1, H=2, D=channels, K=2, Lq=2, seed=3,
                                                   dtype=torch.float64)
    value, loc, attn = (x.to(DEV).requires_grad_(True) for x in (value, loc, attn))
    assert gradcheck(_mod().MSDeformAttnFunction.apply, (value, shp.to(DEV), lsi.to(DEV), loc, attn, 2))


def test_autograd_function_surface():
    m = _mod()
    value, shp, lsi, loc, attn = (x.to(DEV) for x in synth.msda_inputs(((6, 4), (3, 2)), H=2, D=32, K=2, Lq=3))
    value.requires_grad_(True), loc.requires_grad_(True), attn.requires_grad_(True)
    out = m.MSDeformAttnFunction.apply(value, shp, lsi, loc, attn, 64)
    out.sum().backward()
    assert value.grad.shape == value.shape and loc.grad.shape == loc.shape and attn.grad.shape == attn.shape
    assert shp.grad is None and lsi.grad is None


def test_module_matches_oracle_module():
    """MSDeformAttn (nn.Module mirror) against the functional oracle of modules/ms_deform_attn.py:88-130."""
    from memotr_b200.ms_deform_attn import MSDeformAttn
    from oracle import frame as oframe
    torch.manual_seed(0)
    mod = MSDeformAttn(256, 4, 8, 4)
    with torch.no_grad():
        mod.sampling_offsets.weight.normal_(0, 0.02)
        mod.attention_weights.weight.normal_(0, 0.05)
    shapes = synth.SMALL_SHAPES
    S = sum(h * w for h, w in shapes)
    g = torch.Generator().manual_seed(5)
    query, src = torch.randn(2, 7, 256, generator=g), torch.randn(2, S, 256, generator=g)
    mask = torch.zeros(2, S, dtype=torch.bool)
    mask[1, -9:] = True
    shp = torch.as_tensor(shapes, dtype=torch.long)
    lsi = torch.cat((shp.new_zeros(1), shp.prod(1).cumsum(0)[:-1]))
    for ref in (torch.rand(2, 7, 4, 2, generator=g), torch.rand(2, 7, 4, 4, generator=g) * 0.5 + 0.2):
        sd = {"m." + k: v for k, v in mod.state_dict().items()}
        with torch.no_grad():
            want = oframe.msda_module(sd, "m", query, ref, src, shapes, lsi, mask, 8, 4, 4)
            got = mod.to(DEV)(query.to(DEV), ref.to(DEV), src.to(DEV), shp.to(DEV), lsi.to(DEV), mask.to(DEV))
        assert rel_err(got.cpu().numpy(), want.numpy()) < 1e-4
        mod.cpu()
