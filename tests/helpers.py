"""Shared test helpers: rebuild the exact synthetic checkpoint + inputs of a golden case."""
import os

import numpy as np
import torch

from ezaudio_b200 import synth, weights

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

DIT_CASES = {
    # name: (cfg factory, kwargs)
    "dit_tiny72": (lambda: synth.tiny_model(72), dict(B=2, L=40, Lc=12, seed=3, inpaint=False)),
    "dit_tiny72_inpaint": (lambda: synth.tiny_model(72), dict(B=3, L=52, Lc=12, seed=3, inpaint=True)),
    "dit_tiny64": (lambda: synth.tiny_model(64, heads=4, depth=2), dict(B=2, L=130, Lc=100, seed=4, inpaint=False)),
    "dit_L_c1": (lambda: synth.model_cfg("l"), dict(B=1, L=256, Lc=100, seed=1, inpaint=False)),
    "dit_XL": (lambda: synth.model_cfg("xl"), dict(B=2, L=500, Lc=100, seed=2, inpaint=False)),
    "dit_XL_inpaint_30s": (lambda: synth.model_cfg("xl"), dict(B=2, L=1500, Lc=100, seed=2, inpaint=True)),   # BASELINE config C5 shapes
}


def checksum(sd):
    return float(sum(v.double().abs().sum() for v in sd.values()))


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def sampled(x, g):
    """The entries of a full output `x` that golden `g` stores: config-scale goldens keep every `out_stride`-th entry of the last axis."""
    return x[..., ::int(g["out_stride"])] if "out_stride" in g.files else x


def dit_case_inputs(name):
    """-> cfg, sd, dict(x, t, ctx, mask, gt, gt_mask), golden npz."""
    mk, kw = DIT_CASES[name]
    cfg = mk()
    g = load_golden(name)
    sd = weights.synthetic_state_dict(weights.dit_param_shapes(cfg), kw["seed"])
    assert abs(checksum(sd) - float(g["sd_checksum"])) <= 1e-6 * float(g["sd_checksum"]), "synthetic weights differ from golden run"
    B, L, Lc = kw["B"], kw["L"], kw["Lc"]
    x = synth.synth_latents(B, L)
    ctx, mask = synth.synth_context(B, Lc, cfg["context_dim"])
    if B > 1:
        mask[-1] = False
        mask[-1, 0] = True
    t = torch.from_numpy(g["t"])
    gt, gm = synth.synth_gt(B, L) if kw["inpaint"] else (None, None)
    return cfg, sd, dict(x=x, t=t, ctx=ctx, mask=mask, gt=gt, gt_mask=gm), g
