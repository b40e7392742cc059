"""LayerNorm folded into the neighbouring GEMMs (csrc/gemm.cuh FoldIn / FoldOut; option "ln_fold", read when a handle is created).

With the fold ON no LayerNorm kernel is launched on the fast (bf16) path when the whole batch shares one timestep: the GEMM that writes the
residual stream also writes bf16(x * g) and per-row partial sums, the GEMM behind the LayerNorm applies rstd * (acc - mu * u) + v in its
epilogue.  Same tolerances as the unfolded fast mode (tests/test_dit_gpu.py): < 6e-2 max / 1.2e-2 mean against the UNMODIFIED reference's
goldens; per-sample timesteps fall back to the LayerNorm kernels and must still be right."""
import contextlib

import pytest
import torch

from ezaudio_b200 import synth, weights
from tests import helpers

pytestmark = pytest.mark.gpu


@contextlib.contextmanager
def fold_option(v):
    from ezaudio_b200 import _lib
    L = _lib.lib()
    _lib.check(L.ezb_set_option(b"ln_fold", int(v)))
    try:
        yield
    finally:
        _lib.check(L.ezb_set_option(b"ln_fold", FOLD_DEFAULT))


FOLD_DEFAULT = 0


def _launches():
    from ezaudio_b200 import _lib
    return int(_lib.lib().ezb_launch_count())


@pytest.mark.parametrize("name", ["dit_tiny72", "dit_tiny64", "dit_L_c1", "dit_XL", "dit_tiny72_inpaint", "dit_XL_inpaint_30s"])
def test_dit_folded_matches_reference(name):
    from ezaudio_b200.dit import MaskDiT
    cfg, sd, inp, g = helpers.dit_case_inputs(name)
    B, _, L = inp["x"].shape
    outs, counts = {}, {}
    for fold in (0, 1):
        with fold_option(fold):
            m = MaskDiT(precision="bf16", max_batch=B, max_len=L, max_ctx_len=inp["ctx"].shape[1], max_timesteps=8, **cfg).load_state_dict(sd)
        gt = None if inp["gt"] is None else inp["gt"].cuda()
        gm = None if inp["gt_mask"] is None else inp["gt_mask"].cuda()
        args = (inp["x"].cuda(), inp["t"], inp["ctx"].cuda())
        m(*args, context_mask=inp["mask"].cuda(), gt=gt, mae_mask_infer=gm)   # tables, tensor maps
        n0 = _launches()
        out, _ = m(*args, context_mask=inp["mask"].cuda(), gt=gt, mae_mask_infer=gm)
        torch.cuda.synchronize()
        counts[fold] = _launches() - n0
        outs[fold] = out.cpu()
    ref = torch.from_numpy(g["out"])
    err = (helpers.sampled(outs[1], g) - ref).abs()
    print(f"[parity] {name} [bf16, LayerNorm folded]: max-abs {float(err.max()):.3e} mean-abs {float(err.mean()):.3e}; launches {counts[1]} vs {counts[0]} unfolded; "
          f"folded vs unfolded max-abs {float((outs[1] - outs[0]).abs().max()):.3e}")
    assert float(err.max()) < 6e-2 and float(err.mean()) < 1.2e-2
    uniform = inp["t"].dim() == 0 or bool((inp["t"] == inp["t"].flatten()[0]).all())
    nblk = cfg["depth"] + 1
    if uniform:   # 3 LayerNorms per block + skip norms + final norm are gone
        assert counts[0] - counts[1] == 3 * nblk + cfg["depth"] // 2 + 1, counts
    else:
        assert counts[0] == counts[1], counts


@pytest.mark.parametrize("name", ["controlnet_tiny72", "controlnet_XL"])
def test_controlnet_folded_matches_reference(name):
    """ControlNet handle (block outputs feed the next norm1 AND the zero-linears) + out-blocks taking controlnet skips (skip_norm falls back to
    the LayerNorm kernel there, every other LayerNorm stays folded)."""
    from ezaudio_b200.dit import DiTControlNet, MaskDiT
    xl = name.endswith("XL")
    cfg, cn = (synth.model_cfg("xl") if xl else synth.tiny_model(72)), synth.CONTROLNET
    g = helpers.load_golden(name)
    seed, stride = int(g["seed"]), (int(g["skip_stride"]) if "skip_stride" in g.files else 1)
    sd = weights.synthetic_state_dict(weights.dit_param_shapes(cfg), seed)
    sd_cn = weights.synthetic_state_dict(weights.controlnet_param_shapes(cfg, cn), seed + 1)
    B, L, Lc = 2, int(g["L"]), int(g["Lc"])
    x = synth.synth_latents(B, L).cuda()
    ctx, mask = synth.synth_context(B, Lc, cfg["context_dim"])
    ctx, mask = ctx.cuda(), mask.cuda()
    cond = torch.rand(B, 1, 2 * L, generator=torch.Generator().manual_seed(9)).cuda()
    t = torch.tensor(499)
    kw = dict(precision="bf16", max_batch=B, max_len=L, max_ctx_len=Lc, max_timesteps=8)
    with fold_option(1):
        unet = MaskDiT(**kw, **cfg).load_state_dict(sd)
        cnet = DiTControlNet(**kw, **cfg, **cn).load_state_dict(sd_cn, mask_embed=sd["mask_embed"])
    x257, _ = unet(x, t, ctx, context_mask=mask, forward_model=False)
    skips = cnet(x257, t, ctx, context_mask=mask, condition=cond, conditioning_scale=0.8)
    out = unet.model(x257, t, ctx, context_mask=mask, controlnet_skips=list(skips))
    torch.cuda.synchronize()
    s0, s1 = torch.from_numpy(g["skip0"]), torch.from_numpy(g["skip_last"])
    e0 = float((skips[0][:, ::stride].cpu() - s0).abs().max())
    e1 = float((skips[-1][:, ::stride].cpu() - s1).abs().max())
    eo = float((out.cpu() - torch.from_numpy(g["out"])).abs().max())
    print(f"[parity] {name} [bf16, LayerNorm folded]: skip0 {e0:.3e} skip_last {e1:.3e} (std {float(s1.std()):.2f}) out {eo:.3e}")
    assert e0 < 6e-2 * max(1.0, float(s0.std())) and e1 < 6e-2 * max(1.0, float(s1.std())) and eo < 6e-2


def test_loop_graphs_and_short_clips_with_fold():
    """Sampling loop with the fold: graph replay == eager bit for bit (fixed-order partial sums: deterministic), result close to the unfolded
    loop and to the fp32 oracle loop; clips of 25 frames (a warp's 32 rows span clip boundaries)."""
    from ezaudio_b200.dit import MaskDiT
    from ezaudio_b200.inference import sample_latents
    from ezaudio_b200.scheduler import DDIMScheduler
    from oracle import ezaudio_oracle as O
    cfg = synth.tiny_model(72)
    sd = weights.synthetic_state_dict(weights.dit_param_shapes(cfg), 3)
    for B, L, Lc, steps in ((2, 40, 12, 4), (3, 25, 12, 3)):
        ctx, mask = synth.synth_context(B, Lc, cfg["context_dim"])
        uctx, umask = synth.synth_context(1, Lc, cfg["context_dim"], seed=8, uncond=True)
        noise = synth.synth_latents(B, L, seed=5)
        gen = torch.Generator().manual_seed(9)
        step_noise = [torch.randn(B, 128, L, generator=gen) for _ in range(steps)]
        with torch.no_grad():
            ref = O.sample_loop(sd, cfg, noise, ctx, mask, uctx.expand(B, -1, -1), umask.expand(B, -1), guidance_scale=5.0, guidance_rescale=0.75,
                                ddim_steps=steps, eta=1.0, step_noise=step_noise)
        kw = dict(audio_frames=L, guidance_scale=5.0, guidance_rescale=0.75, ddim_steps=steps, eta=1.0, init_noise=noise,
                  step_noise=[s.cuda() for s in step_noise])
        res = {}
        for fold in (0, 1):
            with fold_option(fold):
                m = MaskDiT(precision="bf16", max_batch=2 * B, max_len=L, max_ctx_len=Lc, max_timesteps=8, **cfg).load_state_dict(sd)
            a = sample_latents(m, DDIMScheduler(), ctx, mask, uctx, umask, **kw)
            b = sample_latents(m, DDIMScheduler(), ctx, mask, uctx, umask, **kw)                      # graph replay
            c = sample_latents(m, DDIMScheduler(), ctx, mask, uctx, umask, use_graphs=False, **kw)    # eager again
            assert torch.equal(a, b) and torch.equal(a, c), fold
            res[fold] = a.cpu()
        e_ref, e_pair = float((res[1] - ref).abs().max()), float((res[1] - res[0]).abs().max())
        print(f"[parity] {steps}-step loop B{B} L{L} [bf16, LayerNorm folded]: vs oracle {e_ref:.3e}, vs unfolded {e_pair:.3e}")
        assert e_ref < 0.25 and e_pair < 0.25


DEFAULTS = {"ln_fold": FOLD_DEFAULT, "attn6": 5, "attn_pp": 0, "dhp80": 1, "heads_direct": 0, "ln_tail": 0, "mlp_fused": 0, "ln_variant": 2, "ksub2": 1, "cq_single": 0, "mlp2_pair": 0,
            "attn_res": 0, "w_prefetch": 0, "attn7": 0}


@contextlib.contextmanager
def options(**kw):
    from ezaudio_b200 import _lib
    L = _lib.lib()
    for k, v in kw.items():
        _lib.check(L.ezb_set_option(k.encode(), int(v)))
    try:
        yield
    finally:
        for k in kw:
            _lib.check(L.ezb_set_option(k.encode(), DEFAULTS[k]))


OPTION_SETS = [("heads_direct", dict(heads_direct=1)), ("dhp128", dict(dhp80=0)), ("attn_gen4", dict(attn6=0)), ("all", dict(attn6=7, dhp80=1, heads_direct=1, ln_fold=1)),
               ("ln_tail", dict(ln_tail=1)), ("ln_variant1", dict(ln_variant=1)), ("mlp_fused", dict(mlp_fused=1)), ("mlp_fused+ln_tail+dhp80", dict(mlp_fused=1, ln_tail=1, dhp80=1)),
               ("attn_gen4_token", dict(attn6=0, attn_pp=1)), ("ksub2_qkv", dict(ksub2=3)), ("ksub2_off", dict(ksub2=0)), ("ln_variant0", dict(ln_variant=0)),
               ("cq_single", dict(cq_single=1)), ("mlp2_pair", dict(mlp2_pair=1)), ("attn_gen4_res", dict(attn6=0, attn_res=1)), ("attn6_plain", dict(attn6=1)),
               ("attn6_token", dict(attn6=3)), ("w_prefetch", dict(w_prefetch=1)), ("attn7", dict(attn7=1))]
# every option set on the tiny models and on EzAudio-XL (the benchmarked configuration); the two other large goldens (30-s inpainting: L = 1500, 12 key tiles;
# EzAudio-L: dh = 64) only with the sets that change what those shapes exercise -- the full cross product costs 8 GPU-minutes of weight loading
HEAVY_KEYS = {"attn_gen4", "all", "mlp_fused", "attn6_plain", "attn7", "ksub2_off"}
OPTION_CASES = [pytest.param(name, opts, id=f"{name}-{oid}") for oid, opts in OPTION_SETS
                for name in ("dit_tiny72", "dit_tiny64", "dit_tiny72_inpaint", "dit_XL", "dit_XL_inpaint_30s", "dit_L_c1")
                if name not in ("dit_XL_inpaint_30s", "dit_L_c1") or oid in HEAVY_KEYS]


@pytest.mark.parametrize("name,opts", OPTION_CASES)
def test_fast_path_options_keep_parity(name, opts):
    """Every fast-path variant behind a runtime switch (q/k epilogue without smem staging, 80-element q/k rows, attention generations 4 / 6 and their modes, folded LayerNorm)
    holds the fast mode's tolerance against the reference goldens, alone and all together."""
    from ezaudio_b200.dit import MaskDiT
    cfg, sd, inp, g = helpers.dit_case_inputs(name)
    B, _, L = inp["x"].shape
    with options(**opts):
        m = MaskDiT(precision="bf16", max_batch=B, max_len=L, max_ctx_len=inp["ctx"].shape[1], max_timesteps=8, **cfg).load_state_dict(sd)
        gt = None if inp["gt"] is None else inp["gt"].cuda()
        gm = None if inp["gt_mask"] is None else inp["gt_mask"].cuda()
        out, _ = m(inp["x"].cuda(), inp["t"], inp["ctx"].cuda(), context_mask=inp["mask"].cuda(), gt=gt, mae_mask_infer=gm)
        torch.cuda.synchronize()
        if "w_prefetch" in opts:   # the first pass records the order of the weight reads, the second one issues the L2 prefetch hints: same bits
            out2, _ = m(inp["x"].cuda(), inp["t"], inp["ctx"].cuda(), context_mask=inp["mask"].cuda(), gt=gt, mae_mask_infer=gm)
            torch.cuda.synchronize()
            assert torch.equal(out, out2)
    err = (helpers.sampled(out.cpu(), g) - torch.from_numpy(g["out"])).abs()
    print(f"[parity] {name} [bf16, {opts}]: max-abs {float(err.max()):.3e} mean-abs {float(err.mean()):.3e}")
    assert float(err.max()) < 6e-2 and float(err.mean()) < 1.2e-2


def test_ln_tail_bit_identical_and_controlnet():
    """LayerNorm as the tail phase of the GEMM that produces its input (gemm_ln.cuh): the same arithmetic as the stand-alone kernels, so the
    DiT output must be BIT-IDENTICAL with and without it -- on XL (M = 1000 tokens: every residual-stream GEMM is a one-wave swap-AB launch),
    with ControlNet skips (the skip_norm tail adds the ControlNet skip) and through the graph-replayed sampling loop."""
    from ezaudio_b200.dit import DiTControlNet, MaskDiT
    from ezaudio_b200.inference import sample_latents
    from ezaudio_b200.scheduler import DDIMScheduler
    cfg, cn = synth.model_cfg("xl"), synth.CONTROLNET
    g = helpers.load_golden("controlnet_XL")
    seed = int(g["seed"])
    sd = weights.synthetic_state_dict(weights.dit_param_shapes(cfg), seed)
    sd_cn = weights.synthetic_state_dict(weights.controlnet_param_shapes(cfg, cn), seed + 1)
    B, L, Lc = 2, int(g["L"]), int(g["Lc"])
    x = synth.synth_latents(B, L).cuda()
    ctx, mask = synth.synth_context(B, Lc, cfg["context_dim"])
    ctx, mask = ctx.cuda(), mask.cuda()
    cond = torch.rand(B, 1, 2 * L, generator=torch.Generator().manual_seed(9)).cuda()
    t = torch.tensor(499)
    kw = dict(precision="bf16", max_batch=2 * B, max_len=L, max_ctx_len=Lc, max_timesteps=8)
    unet = MaskDiT(**kw, **cfg).load_state_dict(sd)
    cnet = DiTControlNet(**kw, **cfg, **cn).load_state_dict(sd_cn, mask_embed=sd["mask_embed"])
    uctx, umask = synth.synth_context(1, Lc, cfg["context_dim"], seed=8, uncond=True)
    noise = synth.synth_latents(B, L, seed=5)
    res = {}
    for tail in (0, 1):
        with options(ln_tail=tail, ln_variant=0):   # the tail runs the plain (w, b, scale, shift) LayerNorm arithmetic: compare against that kernel
            x257, _ = unet(x, t, ctx, context_mask=mask, forward_model=False)
            skips = cnet(x257, t, ctx, context_mask=mask, condition=cond, conditioning_scale=0.8)
            out = unet.model(x257, t, ctx, context_mask=mask, controlnet_skips=list(skips))
            plain, _ = unet(x, t, ctx, context_mask=mask)
            lat = sample_latents(unet, DDIMScheduler(), ctx.cpu(), mask.cpu(), uctx, umask, audio_frames=L, guidance_scale=5.0, guidance_rescale=0.75,
                                 ddim_steps=2, eta=0, init_noise=noise)
            lat2 = sample_latents(unet, DDIMScheduler(), ctx.cpu(), mask.cpu(), uctx, umask, audio_frames=L, guidance_scale=5.0, guidance_rescale=0.75,
                                  ddim_steps=2, eta=0, init_noise=noise)   # graph replay
            torch.cuda.synchronize()
            assert torch.equal(lat, lat2)
            res[tail] = (out.clone(), plain.clone(), skips[-1].clone(), lat.clone())
    for a, b in zip(res[0], res[1]):
        assert torch.equal(a, b)
    assert float((res[1][0].cpu() - torch.from_numpy(g["out"])).abs().max()) < 6e-2
