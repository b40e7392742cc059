"""Pins oracle/ezaudio_oracle.py (CPU restatement) against golden outputs of the UNMODIFIED
reference modules (tests/golden/*.npz, made by oracle/gen_golden.py).  fp32 both sides: the
only difference is reduction order, so the tolerance is fp32 round-off (2e-4 abs on O(1)
outputs after 29 blocks; measured ~1e-5)."""
import numpy as np
import pytest
import torch

from ezaudio_b200 import synth, weights
from oracle import ezaudio_oracle as O
from tests import helpers

TOL = 2e-4


@pytest.mark.parametrize("name", ["dit_tiny72", "dit_tiny72_inpaint", "dit_tiny64", "dit_L_c1",
                                  pytest.param("dit_XL", marks=pytest.mark.slow), pytest.param("dit_XL_inpaint_30s", marks=pytest.mark.slow)])
def test_dit_oracle_matches_reference_golden(name):
    cfg, sd, inp, g = helpers.dit_case_inputs(name)
    with torch.no_grad():
        out, _ = O.maskdit_forward(sd, cfg, inp["x"], inp["t"], inp["ctx"], inp["mask"], inp["gt"], inp["gt_mask"])
    err = float((helpers.sampled(out, g) - torch.from_numpy(g["out"])).abs().max())
    assert err < TOL, err


@pytest.mark.parametrize("name,cfg,seed,L,Lc", [("controlnet_tiny72", synth.tiny_model(72), 5, 40, 12),
                                                pytest.param("controlnet_XL", synth.model_cfg("xl"), 2, 500, 100, marks=pytest.mark.slow)])
def test_controlnet_oracle_matches_reference_golden(name, cfg, seed, L, Lc):
    cn = synth.CONTROLNET
    g = helpers.load_golden(name)
    stride = int(g["skip_stride"]) if "skip_stride" in g.files else 1
    sd = weights.synthetic_state_dict(weights.dit_param_shapes(cfg), seed)
    sd_cn = weights.synthetic_state_dict(weights.controlnet_param_shapes(cfg, cn), seed + 1)
    x = synth.synth_latents(2, L)
    ctx, mask = synth.synth_context(2, Lc, cfg["context_dim"])
    cond = torch.rand(2, 1, 2 * L, generator=torch.Generator().manual_seed(9))
    t = torch.tensor(499)
    with torch.no_grad():
        x257, _ = O.maskdit_forward(sd, cfg, x, t, ctx, mask, forward_model=False)
        skips = O.controlnet_forward(sd_cn, cfg, x257, t, ctx, mask, cond, 0.8)
        out = O.udit_forward(sd, cfg, x257, t, ctx, mask, controlnet_skips=skips)
    assert float((skips[0][:, ::stride] - torch.from_numpy(g["skip0"])).abs().max()) < TOL
    assert float((skips[-1][:, ::stride] - torch.from_numpy(g["skip_last"])).abs().max()) < TOL
    assert float((out - torch.from_numpy(g["out"])).abs().max()) < TOL


@pytest.mark.parametrize("name,dcfg,B,L", [("vae_tiny", synth.tiny_vae(16), 2, 9), ("vae_full", synth.VAE_DECODER, 1, 12),
                                           pytest.param("vae_full_10s", synth.VAE_DECODER, 2, 500, marks=pytest.mark.slow)])
def test_vae_oracle_matches_reference_golden(name, dcfg, B, L):
    g = helpers.load_golden(name)
    sd = weights.synthetic_state_dict(weights.vae_decoder_param_shapes(dcfg), 6)
    z = synth.synth_latents(B, L, dcfg["latent_dim"], seed=31)
    with torch.no_grad():
        wav = O.vae_decode(sd, z, strides=tuple(dcfg["strides"]))
    ref = torch.from_numpy(g["out"])
    assert wav.shape == (B, 1, 480 * L)
    wav = helpers.sampled(wav, g)
    assert wav.shape == ref.shape
    assert float((wav - ref).abs().max()) < 1e-5 + 1e-4 * float(ref.abs().max())


def test_ddim_invariants():
    """diffusers is absent (parity unpinned): closed-form checks from SURVEY Appendix B."""
    s = O.DDIM()
    ts = s.set_timesteps(50)
    assert ts.tolist() == list(range(999, 0, -20))
    assert s.set_timesteps(100).tolist() == list(range(999, 0, -10))
    assert float(s.alphas_cumprod[999]) == 0.0
    assert abs(float(s.alphas_cumprod[979]) - 8.5788e-5) < 1e-8
    assert abs(float(s.alphas_cumprod[0]) - 0.99915) < 1e-5
    s.set_timesteps(50)
    x = torch.randn(2, 128, 16, generator=torch.Generator().manual_seed(0))
    v = torch.randn(2, 128, 16, generator=torch.Generator().manual_seed(1))
    # at t=999: a=0 -> x0 = -v, eps = x ; eta=0 -> prev = sqrt(ap)*(-v) + sqrt(1-ap)*x
    ap = s.alphas_cumprod[979]
    assert torch.allclose(s.step(v, 999, x, 0.0), ap.sqrt() * (-v) + (1 - ap).sqrt() * x, atol=1e-6)
    # eta=1: radicand stays >= 0 on every step of the 50- and 100-step schedules
    for n in (50, 100):
        for t in s.set_timesteps(n).tolist():
            a, ap, b, sig = s.coeffs(t, 1.0)
            assert float(1 - ap - sig ** 2) >= 0.0
    # last step lands on final_alpha_cumprod = 1 -> returns x0 when eta = 0
    s.set_timesteps(50)
    a = s.alphas_cumprod[19]
    assert torch.allclose(s.step(v, 19, x, 0.0), a.sqrt() * x - (1 - a).sqrt() * v, atol=1e-6)


def test_cfg_rescale_matches_formula():
    g = torch.Generator().manual_seed(0)
    t, u = torch.randn(3, 128, 20, generator=g), torch.randn(3, 128, 20, generator=g)
    out = O.cfg_combine(t, u, 5.0, 0.75)
    c = u + 5.0 * (t - u)
    want = 0.75 * c * (t.flatten(1).std(1) / c.flatten(1).std(1)).view(-1, 1, 1) + 0.25 * c
    assert torch.allclose(out, want, atol=1e-6)


@pytest.mark.parametrize("name,ecfg,B,L", [("vae_enc_tiny", synth.tiny_vae_encoder(16), 2, 9), ("vae_enc_full", synth.VAE_ENCODER, 1, 12),
                                           pytest.param("vae_enc_full_10s", synth.VAE_ENCODER, 1, 500, marks=pytest.mark.slow)])
def test_vae_encoder_oracle_matches_reference_golden(name, ecfg, B, L):
    g = helpers.load_golden(name)
    sd = weights.synthetic_state_dict(weights.vae_encoder_param_shapes(ecfg), 8)
    audio = 0.3 * torch.randn(B, 1, 480 * L, generator=torch.Generator().manual_seed(41))
    ref = torch.from_numpy(g["out"])  # (B, 256, L): mean | scale
    with torch.no_grad():
        mean = O.vae_encode(sd, audio, None, strides=tuple(ecfg["strides"]))
        noise = torch.randn(B, 128, L, generator=torch.Generator().manual_seed(5))
        z = O.vae_encode(sd, audio, noise, strides=tuple(ecfg["strides"]))
    tol = 1e-5 + 1e-4 * float(ref.abs().max())
    assert float((mean - ref[:, :128]).abs().max()) < tol
    want = noise * (torch.nn.functional.softplus(ref[:, 128:]) + 1e-4) + ref[:, :128]   # bottleneck.py:66-70
    assert float((z - want).abs().max()) < 10 * tol


@pytest.mark.parametrize("name,kw", [("energy_api", dict(hop_size=240, window_size=1920, min_db=-60.0, norm=True)),
                                     ("energy_quant", dict(hop_size=512, window_size=1024, min_db=-80.0, norm=True, quantize_levels=16))])
def test_energy_oracle_matches_reference_golden(name, kw):
    """EnergyExtractor of the unmodified reference (src/models/conditions/energy.py) vs the oracle's restatement."""
    g = helpers.load_golden(name)
    audio = synth.synth_energy_audio(int(g["B"]), int(g["T"]), int(g["seed"]))
    assert abs(float(audio.double().abs().sum()) - float(g["audio_checksum"])) < 1e-6 * float(g["audio_checksum"])
    out = O.energy_extract(audio, **kw)
    assert out.shape == g["out"].shape
    assert float((out - torch.from_numpy(g["out"])).abs().max()) < 2e-5


@pytest.mark.parametrize("name,cfg,B,L,seed", [("t5_tiny", synth.tiny_t5(), 3, 20, 12), ("t5_tiny_h3", synth.tiny_t5(d_kv=32, heads=6, layers=3), 2, 100, 13),
                                               ("t5_large", synth.T5_LARGE, 2, 100, 14)])
def test_t5_oracle_matches_transformers_golden(name, cfg, B, L, seed):
    """T5 encoder restatement vs transformers.T5EncoderModel (5.5.0, the class the reference instantiates) on the synthetic checkpoint."""
    g = helpers.load_golden(name)
    sd = weights.synthetic_state_dict(weights.t5_param_shapes(cfg), seed)
    ids, mask = synth.synth_tokens(B, L, cfg["vocab_size"])
    assert int(ids.sum()) == int(g["ids_checksum"])
    with torch.no_grad():
        out = O.t5_encode(sd, cfg, ids, mask)
    ref = torch.from_numpy(g["out"])
    assert out.shape == ref.shape
    assert float((out - ref).abs().max()) < 2e-4
