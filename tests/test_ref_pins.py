"""Pins of the CPU oracle — and of the CUDA path — to the REFERENCE'S OWN CODE.

tests/golden/ref_*.npz hold the outputs of the unmodified reference sources (f5_tts_mlx/*.py) executed on
tests/mlx_shim (torch-backed stand-ins for the MLX / einx primitives; generator:
tests/golden/make_ref_golden.py, run where a checkout of the reference is available).  Here:

  * not-gpu: the oracle must reproduce every fixture to 1e-5 relative L2 (fp32 both sides; integer /
    boolean results bit-exact; log-mel to 1e-4 absolute — the reference builds its filterbank from fp32
    `linspace`s whose last-bit differences are amplified by the slope division);
  * not-gpu: a subset of the fixtures agrees with a separately recorded run of the reference
    (ref_recomputed.npz: the committed numbers really are what the reference computes);
  * gpu: the CUDA path against the same fixtures, inside the bf16 drift rule of test_gpu_parity.py.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import f5_oracle as O
from helpers import ocfg_of, rel

TOL = 1e-5


def T(a):
    return torch.from_numpy(np.asarray(a))


@pytest.fixture(scope="module")
def gate_w():
    from f5_tts_mlx_b200.weights import GATE_CONFIG, random_dit_weights
    return GATE_CONFIG, random_dit_weights(GATE_CONFIG, seed=1234)


# ------------------------------------------------------------------------------------------------
# oracle vs reference-generated fixtures (CPU)
# ------------------------------------------------------------------------------------------------
def test_oracle_dit_forward_matches_reference_code(gate_w, golden_dir):
    cfg, W = gate_w
    z = np.load(os.path.join(golden_dir, "ref_dit_gate.npz"))
    x, cond, text, t = T(z["x"]), T(z["cond"]), T(z["text"]), T(z["t"])
    assert rel(O.dit_forward(x, cond, text, t, False, False, None, W, ocfg_of(cfg)), T(z["out"])) < TOL
    assert rel(O.dit_forward(x, cond, text, t, True, True, None, W, ocfg_of(cfg)), T(z["out_drop"])) < TOL
    # batch 2, key-padding mask: the reference's `.expand` branch (dit.py:162) run with the shim's opt-in expand
    lens = T(z["lens2"]); n = z["x2"].shape[1]
    mask = torch.arange(n)[None] < lens[:, None]
    got = O.dit_forward(T(z["x2"]), T(z["cond2"]), T(z["text2"]), t, False, False, mask, W, ocfg_of(cfg))
    assert rel(got, T(z["out_b2"])) < TOL


def test_oracle_sample_matches_reference_code(gate_w, golden_dir):
    cfg, W = gate_w
    z = np.load(os.path.join(golden_dir, "ref_sample_gate.npz"))
    cond, text, n = T(z["cond"]), T(z["text"]), int(z["duration"])
    runs = {"euler_cfg": dict(steps=4, method="euler", cfg_strength=2.0, sway_sampling_coef=-1.0, seed=7),
            "midpoint_nocfg": dict(steps=3, method="midpoint", cfg_strength=0.0, sway_sampling_coef=None, seed=7),
            "rk4_cfg": dict(steps=3, method="rk4", cfg_strength=2.0, sway_sampling_coef=-1.0, seed=11)}
    for name, kw in runs.items():
        out, traj = O.sample(cond, text, n, W, ocfg_of(cfg), **kw)
        assert out.shape == z[name + "_out"].shape and traj.shape == z[name + "_traj"].shape
        assert rel(out, T(z[name + "_out"])) < TOL and rel(traj, T(z[name + "_traj"])) < TOL, name
    # requested duration below lens + 1 is raised to it (cfm.py:317), text longer than the conditioning
    out, traj = O.sample(cond, T(z["text_l"]), 10, W, ocfg_of(cfg), steps=3, method="euler", cfg_strength=2.0, seed=3)
    assert out.shape == z["short_out"].shape == (1, 51, 100) and rel(out, T(z["short_out"])) < TOL
    # raw-wave conditioning: mel front-end inside sample() (cfm.py:283-286)
    pcm = np.load(os.path.join(golden_dir, "mel_fixture.npz"))["pcm"]
    wave = torch.from_numpy(pcm.astype(np.float32) / 32768.0)[None]
    out, traj = O.sample(wave, text, 150, W, ocfg_of(cfg), steps=3, method="euler", cfg_strength=2.0, seed=5)
    assert rel(out, T(z["wave_out"])) < 2 * TOL and rel(traj[-1], T(z["wave_traj_last"])) < 2 * TOL


def test_oracle_mel_matches_reference_code(golden_dir):
    z = np.load(os.path.join(golden_dir, "ref_mel.npz"))
    pcm = np.load(os.path.join(golden_dir, "mel_fixture.npz"))["pcm"]
    wave = torch.from_numpy(pcm.astype(np.float32) / 32768.0)
    mel = O.log_mel_spectrogram(wave)
    assert mel.shape == z["mel"].shape == (1, 93, 100)                    # frames-major, last frame dropped
    assert (mel - T(z["mel"])).abs().max().item() < 1e-4
    odd = wave[: int(z["odd_len"])]
    assert (O.log_mel_spectrogram(odd) - T(z["mel_odd"])).abs().max().item() < 1e-4
    assert (O.mel_filters(24000, 1024, 100) - T(z["filters"])).abs().max().item() < 5e-5


def test_oracle_duration_predictor_matches_reference_code(golden_dir):
    from f5_tts_mlx_b200.weights import random_duration_weights
    z = np.load(os.path.join(golden_dir, "ref_duration.npz"))
    dWo = {"duration." + k: v for k, v in random_duration_weights(seed=int(z["weight_seed"])).items()}
    mel, text, lens = T(z["mel"]), T(z["text"]), T(z["lens"])
    assert rel(O.duration_predictor(mel, text, dWo, O.DurationConfig(), lens=lens), T(z["seconds"])) < TOL
    assert rel(O.duration_predictor(mel[:1], text[:1], dWo, O.DurationConfig()), T(z["seconds_nolens"])) < TOL


def test_oracle_operators_and_host_utils_match_reference_code(golden_dir):
    from f5_tts_mlx_b200.weights import DiTConfig, random_dit_weights
    z = np.load(os.path.join(golden_dir, "ref_ops.npz"))
    tiny = DiTConfig(dim=128, depth=1, heads=2, ff_mult=2, text_dim=64, conv_layers=1, text_num_embeds=50)
    W = random_dit_weights(tiny, seed=int(z["weight_seed"]))
    c = ocfg_of(tiny)
    x, xt, t, text = T(z["x"]), T(z["xt"]), T(z["t"]), T(z["text"])
    n = x.shape[1]
    rope = O.rotary_freqs(n)
    P = "transformer.text_embed.text_blocks.layers.0."
    checks = {
        "time_embed": O.timestep_embedding(t, W),
        "grn": O.grn(x, W[P + "grn.gamma"], W[P + "grn.beta"]),
        "convnext": O.convnext_v2_block(xt, W, P),
        "text_embed": O.text_embedding(text, n, False, W, c),
        "text_embed_drop": O.text_embedding(text, n, True, W, c),
        "conv_pos": O.conv_position_embedding(x, W),
        "rope_freqs": rope,
        "rope_q": O.apply_rotary_pos_emb(x[:, None, :, :64], rope),
        "attention_nomask": O.attention(x, None, rope, W, "transformer.transformer_blocks.0.attn.", 2),
        "dit_block": O.dit_block(x, O.timestep_embedding(t, W), None, rope, W, 0, c),
        "freqs_cis": O.precompute_freqs_cis(64, 96),
    }
    for k, v in checks.items():
        assert v.shape == z[k].shape and rel(v, T(z[k])) < TOL, k
    # integer / boolean host utilities: bit-exact
    assert np.array_equal(O.get_pos_embed_indices(torch.zeros(2, dtype=torch.int32), 20, 16).numpy(), z["pos_idx"])
    assert np.array_equal(O.lens_to_mask(torch.tensor([3.0, 7.0, 5.0])).numpy(), z["lens_to_mask"])
    vocab = {ch: i for i, ch in enumerate(" abcdefghijklmnopqrstuvwxyz")}
    assert np.array_equal(O.list_str_to_idx([list("hello w?rld"), list("abc")], vocab).numpy(), z["list_str_to_idx"])
    assert np.array_equal(O.list_str_to_tensor(["héllo", "ab"]).numpy(), z["list_str_to_tensor"])
    # solvers (cfm.py:38-122) on dy/dt = -y + sin(3t) over the sway-warped grid, and the grid itself (cfm.py:377-381)
    tg = O.time_grid(9, -1.0)
    y0 = torch.linspace(-1, 1, 7)
    for nm in ("euler", "midpoint", "rk4"):
        got = getattr(O, f"odeint_{nm}")(lambda tt, y: -y + torch.sin(3 * tt), y0, tg)
        assert rel(got, T(z[f"odeint_{nm}"])) < TOL
    for steps in (2, 8, 32):
        assert (O.time_grid(steps, -1.0) - T(z[f"tgrid_{steps}"])).abs().max().item() < 2e-7


def test_package_host_mirrors_match_reference_code(golden_dir):
    """The product package's host-side mirrors (not the oracle) against the same reference outputs."""
    from f5_tts_mlx_b200 import utils as U
    from f5_tts_mlx_b200.cfm import time_grid
    z = np.load(os.path.join(golden_dir, "ref_ops.npz"))
    assert np.array_equal(U.lens_to_mask(torch.tensor([3.0, 7.0, 5.0])).numpy(), z["lens_to_mask"])
    vocab = {ch: i for i, ch in enumerate(" abcdefghijklmnopqrstuvwxyz")}
    assert np.array_equal(U.list_str_to_idx([list("hello w?rld"), list("abc")], vocab).numpy(), z["list_str_to_idx"])
    assert np.array_equal(U.list_str_to_tensor(["héllo", "ab"]).numpy(), z["list_str_to_tensor"])
    for steps in (2, 8, 32):
        assert (time_grid(steps, -1.0) - T(z[f"tgrid_{steps}"])).abs().max().item() < 2e-7


def test_generate_host_logic_matches_reference_generate(golden_dir, tmp_path):
    """generate.py:113-244 — what the reference's generate() hands to F5TTS.sample (recorded through the shim)
    vs what this package's generate() hands to it: sentence split, "<ref text> <sentence>" assembly, RMS
    normalisation to 0.1, duration conversion, forwarded keywords.  (The multi-sentence + estimate_duration
    duration is the documented deliberate difference, see f5_tts_mlx_b200/generate.py.)"""
    from f5_tts_mlx_b200 import generate as G
    rec = json.load(open(os.path.join(golden_dir, "ref_generate_calls.json")))
    assert G.split_sentences(rec["gen_text"]) == rec["split"]
    pcm = np.load(os.path.join(golden_dir, "mel_fixture.npz"))["pcm"] // rec["pcm_divisor"]
    G.write_wav(str(tmp_path / "ref.wav"), torch.from_numpy(pcm.astype(np.float32) / 32768.0))
    calls = []

    class Rec:
        _duration_predictor = None
        _vocoder = staticmethod(lambda mel: mel)      # generate() refuses a model without a vocoder

        class transformer:
            device = torch.device("cpu")

        def sample(self, audio, text, duration, **kw):
            calls.append(dict(text="".join(text[0]), duration=-1 if duration is None else int(duration),
                              audio_len=audio.shape[1], audio_rms=float(audio.pow(2).mean().sqrt()),
                              **{k: v for k, v in kw.items() if k in ("steps", "method", "speed", "seed")}))
            return torch.zeros(audio.shape[1] + 2560), None

    G.generate(rec["gen_text"], ref_audio_path=str(tmp_path / "ref.wav"), ref_audio_text="A reference.", steps=4,
               method="euler", estimate_duration=True, speed=1.25, seed=3, f5tts=Rec())
    G.generate("Only one sentence here", ref_audio_path=str(tmp_path / "ref.wav"), ref_audio_text="A reference.",
               duration=2.5, f5tts=Rec())
    assert len(calls) == len(rec["calls"]) == 6
    for i, (mine, theirs) in enumerate(zip(calls, rec["calls"])):
        for k in ("text", "audio_len", "steps", "method", "speed", "seed"):
            assert mine.get(k) == theirs.get(k), (i, k, mine, theirs)
        assert abs(mine["audio_rms"] - theirs["audio_rms"]) < 1e-4
    assert calls[5]["duration"] == rec["calls"][5]["duration"] == int(2.5 * 93.75)   # single-generation path
    # reference: whole-text estimate for sentence 1, then x93.75 per sentence (clipped to 4096 inside sample)
    assert rec["calls"][0]["duration"] == 576 and rec["calls"][1]["duration"] == int(576 * 93.75)
    assert all(93 < c["duration"] < 400 for c in calls[:5])                       # ours: per-sentence estimates


def test_fixtures_are_what_the_reference_code_computes_today(golden_dir):
    """The fixtures against a second run of the unmodified reference on the shim (ref_recomputed.npz, written by
    tests/golden/make_ref_recomputed.py): a fresh DiT forward, F5TTS.sample and log_mel_spectrogram agree to 1e-6."""
    r = np.load(os.path.join(golden_dir, "ref_recomputed.npz"))
    z = np.load(os.path.join(golden_dir, "ref_dit_gate.npz"))
    assert rel(T(r["dit_out"]), T(z["out"])) < 1e-6
    # dit.py:162: mx.array has no .expand -> batch > 1 with a mask cannot run upstream (out_b2 uses the shim's expand)
    assert str(r["masked_batch_error"]) == "AttributeError"
    zs = np.load(os.path.join(golden_dir, "ref_sample_gate.npz"))
    assert rel(T(r["sample_midpoint_nocfg_out"]), T(zs["midpoint_nocfg_out"])) < 1e-6
    assert np.abs(r["mel"] - np.load(os.path.join(golden_dir, "ref_mel.npz"))["mel"]).max() < 1e-6


# ------------------------------------------------------------------------------------------------
# CUDA path vs reference-generated fixtures
# ------------------------------------------------------------------------------------------------
def _drift_ok(got, ref_fixture, emu, factor=3.0, cap=2e-2):
    drift = rel(emu, ref_fixture)
    r = rel(got, ref_fixture)
    assert torch.isfinite(got).all() and r < min(max(factor * drift, 2e-3), cap), f"rel {r:.3e} vs drift {drift:.3e}"


@pytest.mark.gpu
def test_cuda_dit_forward_and_sample_vs_reference_fixtures(gate_w, golden_dir):
    from f5_tts_mlx_b200 import F5TTS
    from helpers import make_dit
    cfg, W = gate_w
    model = make_dit(cfg, W)
    dev = "cuda"
    z = np.load(os.path.join(golden_dir, "ref_dit_gate.npz"))
    x, cond, text, t = T(z["x"]), T(z["cond"]), T(z["text"]), T(z["t"])
    emu = O.dit_forward(x, cond, text, t, False, False, None, W, ocfg_of(cfg), O.Precision(True))
    _drift_ok(model(x.to(dev), cond.to(dev), text.to(dev), t, False, False).cpu(), T(z["out"]), emu)
    lens = T(z["lens2"]); n = z["x2"].shape[1]
    mask = torch.arange(n)[None] < lens[:, None]
    emu2 = O.dit_forward(T(z["x2"]), T(z["cond2"]), T(z["text2"]), t, False, False, mask, W, ocfg_of(cfg), O.Precision(True))
    _drift_ok(model(T(z["x2"]).to(dev), T(z["cond2"]).to(dev), T(z["text2"]).to(dev), t, False, False, mask.to(dev)).cpu(),
              T(z["out_b2"]), emu2)
    zs = np.load(os.path.join(golden_dir, "ref_sample_gate.npz"))
    cond, text, n = T(zs["cond"]), T(zs["text"]), int(zs["duration"])
    f5 = F5TTS(model)
    for name, kw in {"euler_cfg": dict(steps=4, method="euler", cfg_strength=2.0, sway_sampling_coef=-1.0, seed=7),
                     "midpoint_nocfg": dict(steps=3, method="midpoint", cfg_strength=0.0, sway_sampling_coef=None, seed=7),
                     "rk4_cfg": dict(steps=3, method="rk4", cfg_strength=2.0, sway_sampling_coef=-1.0, seed=11)}.items():
        out, traj = f5.sample(cond.to(dev), text, n, **kw)          # seed= : the same torch.randn draw as the shim's mx.random
        emu, _ = O.sample(cond, text, n, W, ocfg_of(cfg), prec=O.Precision(True), **kw)
        _drift_ok(out.cpu(), T(zs[name + "_out"]), emu)
        assert traj.shape == zs[name + "_traj"].shape
        assert torch.equal(traj[0].cpu(), T(zs[name + "_traj"])[0])   # identical initial noise
    pcm = np.load(os.path.join(golden_dir, "mel_fixture.npz"))["pcm"]
    wave = torch.from_numpy(pcm.astype(np.float32) / 32768.0)[None]
    out, _ = f5.sample(wave.to(dev), text, 150, steps=3, method="euler", cfg_strength=2.0, seed=5)
    emu, _ = O.sample(wave, text, 150, W, ocfg_of(cfg), steps=3, method="euler", cfg_strength=2.0, seed=5, prec=O.Precision(True))
    _drift_ok(out.cpu(), T(zs["wave_out"]), emu)


@pytest.mark.gpu
def test_cuda_mel_and_duration_vs_reference_fixtures(golden_dir):
    from f5_tts_mlx_b200 import MelSpec
    from f5_tts_mlx_b200.duration import DurationPredictor, DurationTransformer
    from f5_tts_mlx_b200.weights import random_duration_weights
    dev = "cuda"
    z = np.load(os.path.join(golden_dir, "ref_mel.npz"))
    pcm = np.load(os.path.join(golden_dir, "mel_fixture.npz"))["pcm"]
    wave = torch.from_numpy(pcm.astype(np.float32) / 32768.0)
    assert (MelSpec()(wave.to(dev)).cpu() - T(z["mel"])).abs().max().item() < 2e-3
    assert (MelSpec()(wave[: int(z["odd_len"])].to(dev)).cpu() - T(z["mel_odd"])).abs().max().item() < 2e-3
    zd = np.load(os.path.join(golden_dir, "ref_duration.npz"))
    dW = random_duration_weights(seed=int(zd["weight_seed"]))
    pred = DurationPredictor(DurationTransformer(dim=512, depth=8, heads=8, text_dim=512, ff_mult=2, conv_layers=2,
                                                 text_num_embeds=2545), device=dev).load_weights(dW)
    got = pred(T(zd["mel"]).to(dev), T(zd["text"]), lens=T(zd["lens"])).cpu()
    assert rel(got, T(zd["seconds"])) < 2e-2
