"""CUDA Oobleck decoder vs golden outputs of the UNMODIFIED reference decoder (fp32 CPU).
Tolerance is relative to the output scale (random-init outputs have |max| ~ 0.1):
  bf16x3 parity mode: max-abs < 1e-3 * max|ref| + 1e-5 ;  bf16 fast mode: < 6e-2 * max|ref|  -- the reference's own
  bf16-autocast decoder differs from its fp32 output by ~5 % of |max| (SURVEY Appendix C: 1.6e-3 on |max| 0.03)."""
import pytest
import torch

from ezaudio_b200 import synth, weights
from tests import helpers

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("precision,rel", [("bf16x3", 1e-3), ("bf16", 6e-2)])
@pytest.mark.parametrize("name,dcfg,B,L", [("vae_tiny", synth.tiny_vae(16), 2, 9), ("vae_full", synth.VAE_DECODER, 1, 12),
                                           ("vae_full_10s", synth.VAE_DECODER, 2, 500)])   # the 10-s decode bench.py times
def test_vae_decode_matches_reference(name, dcfg, B, L, precision, rel):
    from ezaudio_b200.vae import OobleckDecoder
    g = helpers.load_golden(name)
    sd = weights.synthetic_state_dict(weights.vae_decoder_param_shapes(dcfg), 6)
    dec = OobleckDecoder(precision=precision, max_batch=B, max_latent_len=L, **dcfg).load_state_dict(sd)
    z = synth.synth_latents(B, L, dcfg["latent_dim"], seed=31).cuda()
    wav = dec(z)
    torch.cuda.synchronize()
    ref = torch.from_numpy(g["out"])
    assert wav.shape == (B, 1, 480 * L)
    wav = helpers.sampled(wav.cpu(), g)
    assert wav.shape == ref.shape
    err = float((wav - ref).abs().max())
    print(f"[parity] {name} [{precision}]: max-abs {err:.3e} (|ref|max {float(ref.abs().max()):.3e})")
    assert err < rel * float(ref.abs().max()) + 1e-5, (err, float(ref.abs().max()))


@pytest.mark.parametrize("precision,rel", [("bf16x3", 1e-3), ("bf16", 6e-2)])
@pytest.mark.parametrize("name,cfgs,B,L", [("vae_enc_tiny", (synth.tiny_vae_encoder(16), synth.tiny_vae(16)), 2, 9),
                                           ("vae_enc_full", (synth.VAE_ENCODER, synth.VAE_DECODER), 1, 12),
                                           ("vae_enc_full_10s", (synth.VAE_ENCODER, synth.VAE_DECODER), 1, 500)])
def test_vae_encode_matches_reference(name, cfgs, B, L, precision, rel):
    """OobleckEncoder (strided implicit-GEMM convs) + VAE bottleneck vs the UNMODIFIED reference encoder's golden output
    (mean | scale), with injected noise for the sampling formula (bottleneck.py:66-70)."""
    from ezaudio_b200.vae import OobleckDecoder
    ecfg, dcfg = cfgs
    g = helpers.load_golden(name)
    sd = dict(weights.synthetic_state_dict(weights.vae_decoder_param_shapes(dcfg), 6))
    sd.update(weights.synthetic_state_dict(weights.vae_encoder_param_shapes(ecfg), 8))
    codec = OobleckDecoder(precision=precision, max_batch=B, max_latent_len=L, encoder_cfg=ecfg, **dcfg).load_state_dict(sd)
    audio = 0.3 * torch.randn(B, 1, 480 * L, generator=torch.Generator().manual_seed(41))
    ref = torch.from_numpy(g["out"])
    mean = codec.encode(audio.cuda(), noise=False).cpu()
    scale_ref = float(ref.abs().max())
    assert float((mean - ref[:, :128]).abs().max()) < rel * scale_ref + 1e-5
    noise = torch.randn(B, 128, L, generator=torch.Generator().manual_seed(5))
    z = codec.encode(audio.cuda(), noise=noise.cuda()).cpu()
    want = noise * (torch.nn.functional.softplus(ref[:, 128:]) + 1e-4) + ref[:, :128]
    assert float((z - want).abs().max()) < 4 * rel * scale_ref + 1e-5
