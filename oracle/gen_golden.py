"""Generates tests/golden/*.npz by running the UNMODIFIED reference modules (CPU fp32, imported from the
tree oracle/refimport.py finds) on the deterministic synthetic checkpoint + inputs, and tests/golden/weight_shapes.json.gz
from the reference modules' state dicts.
Run in the build container:  python oracle/gen_golden.py     -- TEST INFRASTRUCTURE."""
import contextlib
import copy
import gzip
import io
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ezaudio_b200 import synth, weights  # noqa: E402
from oracle import refimport  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def checksum(sd):
    return float(sum(v.double().abs().sum() for v in sd.values()))


@torch.no_grad()
def dit_case(ref, name, cfg, B, L, Lc, seed, inpaint, tscalar=None, tvec=None, out_stride=1):
    sd = weights.synthetic_state_dict(weights.dit_param_shapes(cfg), seed)
    m = refimport.build(ref.MaskDiT, sd, **cfg)
    x = synth.synth_latents(B, L)
    ctx, mask = synth.synth_context(B, Lc, cfg["context_dim"])
    if B > 1:  # last row plays the unconditional prompt
        mask[-1] = False
        mask[-1, 0] = True
    t = torch.tensor(tscalar) if tvec is None else torch.tensor(tvec, dtype=torch.long)
    gt, gm = (synth.synth_gt(B, L) if inpaint else (None, None))
    out, mae = m(x, t, ctx, context_mask=mask, gt=None if gt is None else gt.clone(), mae_mask_infer=gm)
    # config-scale cases keep every `out_stride`-th token (a full 30-s XL output is 1.5 MB)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), out=out[..., ::out_stride].numpy(), sd_checksum=checksum(sd),
                        x_checksum=float(x.double().abs().sum()), seed=seed, B=B, L=L, Lc=Lc,
                        inpaint=inpaint, t=t.numpy(), **({"out_stride": out_stride} if out_stride > 1 else {}))
    print(name, tuple(out.shape), float(out.std()), float(out.abs().max()))


@torch.no_grad()
def controlnet_case(ref, name, cfg, B, L, Lc, seed, skip_stride=1):
    cn = synth.CONTROLNET
    sd = weights.synthetic_state_dict(weights.dit_param_shapes(cfg), seed)
    sd_cn = weights.synthetic_state_dict(weights.controlnet_param_shapes(cfg, cn), seed + 1)
    m = refimport.build(ref.MaskDiT, sd, **cfg)
    c = refimport.build(ref.DiTControlNet, sd_cn, **cfg, **cn)
    x = synth.synth_latents(B, L)
    ctx, mask = synth.synth_context(B, Lc, cfg["context_dim"])
    cond = torch.rand(B, 1, 2 * L, generator=torch.Generator().manual_seed(9))
    t = torch.tensor(499)
    x257, _ = m(x, t, ctx, context_mask=mask, forward_model=False)
    skips = c(x257, t, ctx, context_mask=mask, condition=cond, conditioning_scale=0.8)
    out = m.model(x257, t, ctx, context_mask=mask, controlnet_skips=list(skips))
    # config-scale cases keep every `skip_stride`-th token row of the two stored skips (a full XL skip is 4.6 MB)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), out=out.numpy(), skip0=skips[0][:, ::skip_stride].numpy(),
                        skip_last=skips[-1][:, ::skip_stride].numpy(), sd_checksum=checksum(sd) + checksum(sd_cn), seed=seed,
                        B=B, L=L, Lc=Lc, skip_stride=skip_stride)
    print(name, tuple(out.shape), float(out.std()), float(skips[-1].std()))


@torch.no_grad()
def vae_case(ref, name, dcfg, B, L, seed, out_stride=1):
    sd = weights.synthetic_state_dict(weights.vae_decoder_param_shapes(dcfg), seed)
    m = refimport.build(ref.OobleckDecoder, {k[len("decoder."):]: v for k, v in sd.items()}, **dcfg)
    z = synth.synth_latents(B, L, dcfg["latent_dim"], seed=31)
    wav = m(z)
    # config-scale cases keep every `out_stride`-th sample (a full 10-s stereo batch is 1.9 MB); a stride prime to the 480-sample
    # latent hop still visits every phase of the upsampling chain
    np.savez_compressed(os.path.join(OUT, name + ".npz"), out=wav[..., ::out_stride].numpy(), sd_checksum=checksum(sd), seed=seed, B=B, L=L,
                        **({"out_stride": out_stride} if out_stride > 1 else {}))
    print(name, tuple(wav.shape), float(wav.std()), float(wav.abs().max()))


@torch.no_grad()
def vae_enc_case(ref, name, ecfg, B, T, seed):
    """OobleckEncoder output (mean | scale channels) of the unmodified reference; bottleneck sampling is checked by formula."""
    sd = weights.synthetic_state_dict(weights.vae_encoder_param_shapes(ecfg), seed)
    m = refimport.build(ref.OobleckEncoder, {k[len("encoder."):]: v for k, v in sd.items()}, **ecfg)
    audio = 0.3 * torch.randn(B, 1, T, generator=torch.Generator().manual_seed(41))
    out = m(audio)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), out=out.numpy(), sd_checksum=checksum(sd), seed=seed, B=B, T=T)
    print(name, tuple(out.shape), float(out.std()), float(out.abs().max()))


@torch.no_grad()
def energy_case(ref, name, B, T, seed, **kw):
    """EnergyExtractor (src/models/conditions/energy.py) on clips of different loudness, one of them with silent stretches."""
    audio = synth.synth_energy_audio(B, T, seed)
    out = ref.EnergyExtractor(**kw)(audio)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), out=out.numpy(), audio_checksum=float(audio.double().abs().sum()), seed=seed, B=B, T=T,
                        **{k: (v if v is not None else -1) for k, v in kw.items() if k != "padding"})
    print(name, tuple(out.shape), float(out.mean()), float(out.min()))


@torch.no_grad()
def t5_case(ref, name, cfg, B, L, seed):
    """transformers.T5EncoderModel (the text encoder class the reference instantiates, api/ezaudio.py:79) with the synthetic checkpoint."""
    from transformers import T5Config, T5EncoderModel
    sd = weights.synthetic_state_dict(weights.t5_param_shapes(cfg), seed)
    m = T5EncoderModel(T5Config(feed_forward_proj="gated-gelu", tie_word_embeddings=False, dropout_rate=0.0, **cfg)).eval()
    full = dict(sd)
    full["encoder.embed_tokens.weight"] = sd["shared.weight"]
    missing, unexpected = m.load_state_dict(full, strict=False)
    assert not missing and not unexpected, (missing, unexpected)
    ids, mask = synth.synth_tokens(B, L, cfg["vocab_size"])
    out = m(input_ids=ids, attention_mask=mask).last_hidden_state
    np.savez_compressed(os.path.join(OUT, name + ".npz"), out=out.numpy(), sd_checksum=checksum(sd), ids_checksum=int(ids.sum()), seed=seed, B=B, L=L)
    print(name, tuple(out.shape), float(out.std()), float(out.abs().max()))


def weight_shapes(ref, name):
    """State-dict key -> shape of the reference MaskDiT (XL, L) and DiTControlNet (L), built on the meta device."""
    shapes = {}
    for key, cls, kw in (("MaskDiT_xl", ref.MaskDiT, synth.model_cfg("xl")), ("MaskDiT_l", ref.MaskDiT, synth.model_cfg("l")),
                         ("DiTControlNet_l", ref.DiTControlNet, dict(synth.model_cfg("l"), **synth.CONTROLNET))):
        with torch.device("meta"), contextlib.redirect_stdout(io.StringIO()):
            m = cls(**copy.deepcopy(kw))
        shapes[key] = {k: list(v.shape) for k, v in m.state_dict().items()}
    with open(os.path.join(OUT, name + ".json.gz"), "wb") as f:
        f.write(gzip.compress(json.dumps(shapes).encode(), mtime=0))
    print(name, {k: len(v) for k, v in shapes.items()})


def main():
    ref = refimport.import_reference()
    assert ref is not None, "reference tree not found"
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    only = set(sys.argv[1:])
    global dit_case, controlnet_case, vae_case, vae_enc_case, energy_case, t5_case, weight_shapes
    if only:
        def filt(f):
            return lambda ref, name, *a, **k: f(ref, name, *a, **k) if name in only else None
        dit_case, controlnet_case, vae_case, vae_enc_case = filt(dit_case), filt(controlnet_case), filt(vae_case), filt(vae_enc_case)
        energy_case = filt(energy_case)
        t5_case = filt(t5_case)
        weight_shapes = filt(weight_shapes)
    dit_case(ref, "dit_tiny72", synth.tiny_model(72), B=2, L=40, Lc=12, seed=3, inpaint=False, tscalar=999)
    dit_case(ref, "dit_tiny72_inpaint", synth.tiny_model(72), B=3, L=52, Lc=12, seed=3, inpaint=True, tvec=[999, 500, 19])
    dit_case(ref, "dit_tiny64", synth.tiny_model(64, heads=4, depth=2), B=2, L=130, Lc=100, seed=4, inpaint=False, tscalar=259)
    controlnet_case(ref, "controlnet_tiny72", synth.tiny_model(72), B=2, L=40, Lc=12, seed=5)
    vae_case(ref, "vae_tiny", synth.tiny_vae(16), B=2, L=9, seed=6)
    vae_case(ref, "vae_full", synth.VAE_DECODER, B=1, L=12, seed=6)
    vae_enc_case(ref, "vae_enc_tiny", synth.tiny_vae_encoder(16), B=2, T=480 * 9, seed=8)
    vae_enc_case(ref, "vae_enc_full", synth.VAE_ENCODER, B=1, T=480 * 12, seed=8)
    energy_case(ref, "energy_api", B=3, T=24000 * 2, seed=9, hop_size=240, window_size=1920, padding="reflect", min_db=-60, norm=True)
    energy_case(ref, "energy_quant", B=2, T=5000, seed=10, hop_size=512, window_size=1024, padding="reflect", min_db=-80, norm=True,
                quantize_levels=16)
    t5_case(ref, "t5_tiny", synth.tiny_t5(), B=3, L=20, seed=12)
    t5_case(ref, "t5_tiny_h3", synth.tiny_t5(d_kv=32, heads=6, layers=3), B=2, L=100, seed=13)
    t5_case(ref, "t5_large", synth.T5_LARGE, B=2, L=100, seed=14)
    dit_case(ref, "dit_L_c1", synth.model_cfg("l"), B=1, L=256, Lc=100, seed=1, inpaint=False, tscalar=999)  # BASELINE config 1
    dit_case(ref, "dit_XL", synth.model_cfg("xl"), B=2, L=500, Lc=100, seed=2, inpaint=False, tscalar=479)
    # ---- configuration-scale cases (BASELINE configs C4 / C5 and the 10-s codec the benchmark times)
    controlnet_case(ref, "controlnet_XL", synth.model_cfg("xl"), B=2, L=500, Lc=100, seed=2, skip_stride=20)      # C4 shapes (B_eff = 2)
    dit_case(ref, "dit_XL_inpaint_30s", synth.model_cfg("xl"), B=2, L=1500, Lc=100, seed=2, inpaint=True, tvec=[989, 9], out_stride=2)  # C5 shapes
    vae_case(ref, "vae_full_10s", synth.VAE_DECODER, B=2, L=500, seed=6, out_stride=7)
    vae_enc_case(ref, "vae_enc_full_10s", synth.VAE_ENCODER, B=1, T=480 * 500, seed=8)
    weight_shapes(ref, "weight_shapes")


if __name__ == "__main__":
    main()
