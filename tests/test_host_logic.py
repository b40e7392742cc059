"""CPU-only checks: C-ABI exports, scheduler restatement, weight wire format, prompt sharding (gloo, world_size 2)."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "ezb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ezb_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_loads_and_exports_every_declared_symbol():
    from ezaudio_b200 import _lib, build
    build.build()
    L = ctypes.CDLL(_lib.LIB_PATH)
    names = _header_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/ezb200.h but not exported"
    assert set(_lib.EXPORTS) <= set(names)
    assert _lib.lib().ezb_version() >= 1


def test_no_cpu_fallback_without_library(monkeypatch):
    from ezaudio_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libezb200.so")
    with pytest.raises(_lib.EzbError):
        _lib.lib()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "ezaudio_b200")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            assert not re.search(r"^\s*(from|import)\s+oracle", open(os.path.join(pkg, f)).read(), flags=re.M), f


def test_scheduler_matches_oracle_restatement_and_invariants():
    from ezaudio_b200.scheduler import DDIMScheduler
    from oracle import ezaudio_oracle as O
    s, o = DDIMScheduler(), O.DDIM()
    assert torch.equal(s.alphas_cumprod, o.alphas_cumprod)
    assert float(s.alphas_cumprod[-1]) == 0.0
    for n in (50, 100):
        s.set_timesteps(n)
        assert s.timesteps.tolist() == list(range(999, 0, -1000 // n))
        o.set_timesteps(n)
        x = torch.randn(2, 8, 5, generator=torch.Generator().manual_seed(n))
        v = torch.randn(2, 8, 5, generator=torch.Generator().manual_seed(n + 1))
        z = torch.randn(2, 8, 5, generator=torch.Generator().manual_seed(n + 2))
        for t in s.timesteps.tolist()[:: max(1, n // 10)]:
            for eta in (0.0, 1.0):
                c = s.step_coefficients(t, eta)
                x0, eps = c[0] * x - c[1] * v, c[0] * v + c[1] * x
                mine = c[2] * x0 + c[3] * eps + c[4] * z
                assert torch.allclose(mine, o.step(v, t, x, eta, z), atol=2e-6)


def test_weight_wire_format_matches_reference_golden():
    """State-dict keys / shapes the loader expects == those of the unmodified reference MaskDiT (XL, L) and DiTControlNet (L)
    (tests/golden/weight_shapes.json.gz, written by oracle/gen_golden.py)."""
    import gzip
    import json
    from ezaudio_b200 import synth, weights
    with gzip.open(os.path.join(ROOT, "tests", "golden", "weight_shapes.json.gz"), "rt") as f:
        want = {model: {k: tuple(v) for k, v in shapes.items()} for model, shapes in json.load(f).items()}
    assert want["MaskDiT_xl"] == dict(weights.dit_param_shapes(synth.model_cfg("xl")))
    assert want["MaskDiT_l"] == dict(weights.dit_param_shapes(synth.model_cfg("l")))
    assert want["DiTControlNet_l"] == dict(weights.controlnet_param_shapes(synth.model_cfg("l"), synth.CONTROLNET))


def test_shard_range_covers_everything_once():
    from ezaudio_b200.shard import shard_range
    for n in (0, 1, 4, 7, 32, 33):
        for w in (1, 2, 3, 8):
            spans = [shard_range(n, w, r) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            assert max(b - a for a, b in spans) - min(b - a for a, b in spans) <= 1


def _gloo_worker(rank, world, port, n_total, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from ezaudio_b200.shard import gather_waveforms, shard_prompts, shard_range
    prompts = [f"p{i}" for i in range(n_total)]
    mine = shard_prompts(prompts, world, rank)
    a, b = shard_range(n_total, world, rank)
    local = torch.stack([torch.full((6,), float(i)) for i in range(a, b)]) if b > a else torch.zeros(0, 6)
    full = gather_waveforms(local, n_total, dist)
    q.put((rank, mine, full[:, 0].tolist()))
    dist.destroy_process_group()


@pytest.mark.parametrize("n_total", [4, 5])
def test_prompt_sharding_two_ranks_gloo(n_total):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000 + n_total
    ps = [ctx.Process(target=_gloo_worker, args=(r, 2, port, n_total, q)) for r in range(2)]
    [p.start() for p in ps]
    res = sorted(q.get(timeout=120) for _ in range(2))
    [p.join(timeout=60) for p in ps]
    assert res[0][1] + res[1][1] == [f"p{i}" for i in range(n_total)]
    for _, _, col in res:
        assert col == [float(i) for i in range(n_total)]


def test_t5_bucket_table_host_logic_matches_oracle_and_transformers():
    """The (L, L) relative-position bucket table the Python mirror hands to ezb_t5_forward: equal to the oracle's restatement and, when
    transformers is importable, to T5Attention._relative_position_bucket itself (same float32 truncations at the boundaries 16, 32, 64)."""
    import torch
    from ezaudio_b200.t5 import relative_position_buckets
    from oracle import ezaudio_oracle as O
    for L in (1, 7, 100, 300):
        pos = torch.arange(L)
        rp = pos[None, :] - pos[:, None]
        got = relative_position_buckets(L, 32, 128).long()
        assert torch.equal(got, O.t5_relative_position_bucket(rp, 32, 128))
        try:
            from transformers.models.t5.modeling_t5 import T5Attention
        except Exception:
            continue
        assert torch.equal(got, T5Attention._relative_position_bucket(rp, bidirectional=True, num_buckets=32, max_distance=128))
    assert got.min() >= 0 and got.max() <= 31


def test_hash_tokenizer_contract():
    """Stand-in for T5Tokenizer(text, max_length=, padding='max_length', truncation=True, return_tensors='pt') (src/inference.py:39-41)."""
    from ezaudio_b200.api import HashTokenizer
    tok = HashTokenizer(32128)
    out = tok(["a dog barks", "", "x " * 200], max_length=100, padding="max_length", truncation=True, return_tensors="pt")
    assert out.input_ids.shape == (3, 100) and out.attention_mask.sum(1).tolist() == [4, 1, 100]
    assert out.input_ids[1, 0] == 1 and out.input_ids[0, 3] == 1 and out.input_ids[2, 99] == 1          # EOS closes every prompt
    assert int(out.input_ids.max()) < 32128 and int(out.input_ids[0, 4:].abs().sum()) == 0             # pad id 0
    again = tok("a dog barks", max_length=100)
    assert again.input_ids[0].tolist() == out.input_ids[0].tolist()                                     # stable across calls


def test_wav_io_round_trip(tmp_path):
    """save_wav / _load_audio (the I/O either side of the path: t2a_demo.py:13, api/ezaudio.py:146): float32 round trip, int16 input,
    stereo down-mix and 48 k -> 24 k resampling."""
    from scipy.io import wavfile
    from ezaudio_b200.api import _load_audio, save_wav
    t = np.arange(24000) / 24000.0
    x = (0.5 * np.sin(2 * np.pi * 440 * t)).astype(np.float32)
    p = str(tmp_path / "a.wav")
    save_wav(p, (24000, x))
    assert np.array_equal(_load_audio(p, 24000), x)
    wavfile.write(str(tmp_path / "b.wav"), 24000, (x * 32767).astype(np.int16))
    assert np.abs(_load_audio(str(tmp_path / "b.wav"), 24000) - x).max() < 1e-4
    t48 = np.arange(48000) / 48000.0
    st = np.stack([0.5 * np.sin(2 * np.pi * 440 * t48), 0.5 * np.sin(2 * np.pi * 440 * t48)], 1).astype(np.float32)
    wavfile.write(str(tmp_path / "c.wav"), 48000, st)
    y = _load_audio(str(tmp_path / "c.wav"), 24000)
    assert y.shape == (24000,) and np.abs(y[200:-200] - x[200:-200]).max() < 5e-3
