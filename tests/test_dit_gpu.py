"""CUDA DiT forward (through the C-ABI) vs the UNMODIFIED reference's golden outputs (tests/golden, fp32 CPU).

Tolerances (max-abs on outputs of std ~1, |max| ~4):
  * precision 'bf16x3' (split-bf16 operands, fp32-grade):  < 1e-3  -- BASELINE north_star's bound.
  * precision 'bf16'  (plain bf16 tensor-core operands):    < 6e-2  -- the reference's OWN bf16-autocast path differs from
    its fp32 path by 4.4e-2..5.5e-2 max-abs on config 1 (SURVEY 0.3), so this is the noise floor of the dtype; the mean-abs
    error is additionally bounded by 1.2e-2 (reference bf16: 9e-3).
"""
import pytest
import torch

from ezaudio_b200 import synth, weights
from tests import helpers

pytestmark = pytest.mark.gpu

TOL = {"bf16x3": (1e-3, 2e-4), "bf16": (6e-2, 1.2e-2)}


def _run_case(name, precision):
    from ezaudio_b200.dit import MaskDiT
    cfg, sd, inp, g = helpers.dit_case_inputs(name)
    B, _, L = inp["x"].shape
    m = MaskDiT(precision=precision, max_batch=B, max_len=L, max_ctx_len=inp["ctx"].shape[1], max_timesteps=8, **cfg)
    m.load_state_dict(sd)
    dev = "cuda"
    gt = None if inp["gt"] is None else inp["gt"].to(dev)
    gm = None if inp["gt_mask"] is None else inp["gt_mask"].to(dev)
    out, mae = m(inp["x"].to(dev), inp["t"], inp["ctx"].to(dev), context_mask=inp["mask"].to(dev), gt=gt, mae_mask_infer=gm)
    torch.cuda.synchronize()
    ref = torch.from_numpy(g["out"])
    err = (helpers.sampled(out.cpu(), g) - ref).abs()
    assert torch.isfinite(out).all()
    print(f"[parity] {name} [{precision}]: max-abs {float(err.max()):.3e} mean-abs {float(err.mean()):.3e} (ref std {float(ref.std()):.3f})")
    return float(err.max()), float(err.mean())


@pytest.mark.parametrize("name", ["dit_tiny72", "dit_tiny72_inpaint", "dit_tiny64", "dit_L_c1", "dit_XL", "dit_XL_inpaint_30s"])
def test_dit_parity_mode_matches_reference(name):
    mx, mean = _run_case(name, "bf16x3")
    assert mx < TOL["bf16x3"][0] and mean < TOL["bf16x3"][1], (mx, mean)


@pytest.mark.parametrize("name", ["dit_tiny72", "dit_tiny72_inpaint", "dit_tiny64", "dit_L_c1", "dit_XL", "dit_XL_inpaint_30s"])
def test_dit_fast_mode_within_bf16_floor(name):
    mx, mean = _run_case(name, "bf16")
    assert mx < TOL["bf16"][0] and mean < TOL["bf16"][1], (mx, mean)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_long_clip_30s_matches_oracle(precision):
    """C5 shape: L = 1500 latent frames (30 s) - 12 x 12 attention tiles per head, rotary positions up to 1499 - on the tiny dh=72 model,
    inpainting inputs, CFG-style batch with a one-token unconditional row.  Oracle computed here on the host cores."""
    from ezaudio_b200.dit import MaskDiT
    from oracle import ezaudio_oracle as O
    cfg = synth.tiny_model(72)
    B, L, Lc = 2, 1500, 100
    sd = weights.synthetic_state_dict(weights.dit_param_shapes(cfg), 3)
    x = synth.synth_latents(B, L)
    ctx, mask = synth.synth_context(B, Lc, cfg["context_dim"])
    mask[-1] = False
    mask[-1, 0] = True
    gt, gm = synth.synth_gt(B, L)
    t = torch.tensor([999, 19])
    with torch.no_grad():
        want, _ = O.maskdit_forward(sd, cfg, x, t, ctx, mask, gt=gt.clone(), mae_mask_infer=gm)
    m = MaskDiT(precision=precision, max_batch=B, max_len=L, max_ctx_len=Lc, max_timesteps=8, **cfg).load_state_dict(sd)
    got, _ = m(x.cuda(), t.cuda(), ctx.cuda(), context_mask=mask.cuda(), gt=gt.cuda(), mae_mask_infer=gm.cuda())
    err = (got.cpu() - want).abs()
    assert float(err.max()) < TOL[precision][0] and float(err.mean()) < TOL[precision][1], (float(err.max()), float(err.mean()))
