"""Pins the CPU oracle (oracle/f5_oracle.py) against INDEPENDENT library implementations of the
same operators and against the committed golden fixtures.  The reference has no tests or golden
vectors of its own for this path and MLX cannot run here (parity unpinned by the reference), so
these cross-checks are what the oracle's credibility rests on.  CPU only."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import f5_oracle as O
from f5_tts_mlx_b200.weights import GATE_CONFIG, VocosConfig, random_dit_weights, random_vocos_weights
from helpers import ocfg_of, rel, synth_audio

torch.set_num_threads(max(1, (os.cpu_count() or 2) // 2))


# ---------------- audio front-end ----------------
def test_mel_matches_torchaudio_with_zero_padding_and_dropped_last_frame():
    torchaudio = pytest.importorskip("torchaudio")
    x = synth_audio(24000 * 2 + 123, seed=3)
    ms = torchaudio.transforms.MelSpectrogram(sample_rate=24000, n_fft=1024, win_length=1024, hop_length=256, n_mels=100,
                                              power=1, center=True, pad_mode="constant", norm=None, mel_scale="htk")
    ref = ms(x).clamp(min=1e-5).log().T[:-1]           # reference drops the last frame (audio.py:203)
    got = O.log_mel_spectrogram(x)[0]
    assert got.shape == ref.shape == (x.numel() // 256, 100)
    assert (got - ref).abs().max().item() < 5e-4


def test_mel_filterbank_matches_torchaudio():
    torchaudio = pytest.importorskip("torchaudio")
    fb = torchaudio.functional.melscale_fbanks(513, 0.0, 12000.0, 100, 24000, norm=None, mel_scale="htk")
    assert torch.allclose(O.mel_filters(24000, 1024, 100), fb.T, atol=1e-6)


def test_hann_is_periodic():
    assert torch.allclose(O.hanning(1024), torch.hann_window(1024, periodic=True), atol=1e-7)


def test_mel_golden_fixture(golden_dir):
    z = np.load(os.path.join(golden_dir, "mel_fixture.npz"))
    x = torch.from_numpy(z["pcm"].astype(np.float32) / 32768.0)
    got = O.log_mel_spectrogram(x)[0].numpy()
    assert got.shape == z["mel"].shape == (93, 100)
    np.testing.assert_allclose(got, z["mel"], atol=2e-5)
    # the whole reference clip (wave module: 127985 samples) -> 499 frames (SURVEY §2 #16)
    assert int(z["full_clip_samples"]) == 127985 and int(z["full_clip_frames"]) == 499


@pytest.mark.parametrize("L", [256, 700, 1024, 5000])
def test_mel_frame_count_edge_lengths(L):
    assert O.log_mel_spectrogram(torch.randn(L)).shape == (1, L // 256, 100)


# ---------------- rope / attention / activations ----------------
def test_rope_equals_complex_rotation():
    n, h = 50, 3
    t = torch.randn(1, h, n, 64)
    got = O.apply_rotary_pos_emb(t, O.rotary_freqs(n, 64))
    inv = 1.0 / (10000.0 ** (torch.arange(0, 64, 2).float() / 64))
    ang = torch.arange(n).float()[:, None] * inv[None]
    z = torch.view_as_complex(t.reshape(1, h, n, 32, 2).contiguous()) * torch.polar(torch.ones_like(ang), ang)
    assert torch.allclose(got, torch.view_as_real(z).reshape(1, h, n, 64), atol=1e-5)


def test_attention_matches_sdpa_with_key_padding_mask():
    cfg = GATE_CONFIG
    W = random_dit_weights(cfg, seed=5)
    p = "transformer.transformer_blocks.0.attn."
    b, n = 2, 70
    x = torch.randn(b, n, cfg.dim)
    lens = torch.tensor([70, 41]); mask = torch.arange(n)[None] < lens[:, None]
    rope = O.rotary_freqs(n, 64)
    got = O.attention(x, mask, rope, W, p, cfg.heads)
    q = F.linear(x, W[p + "to_q.weight"], W[p + "to_q.bias"]).view(b, n, cfg.heads, 64).transpose(1, 2)
    k = F.linear(x, W[p + "to_k.weight"], W[p + "to_k.bias"]).view(b, n, cfg.heads, 64).transpose(1, 2)
    v = F.linear(x, W[p + "to_v.weight"], W[p + "to_v.bias"]).view(b, n, cfg.heads, 64).transpose(1, 2)
    q, k = O.apply_rotary_pos_emb(q, rope), O.apply_rotary_pos_emb(k, rope)
    o = F.scaled_dot_product_attention(q, k, v, attn_mask=mask[:, None, None, :])
    o = F.linear(o.transpose(1, 2).reshape(b, n, -1), W[p + "to_out.layers.0.weight"], W[p + "to_out.layers.0.bias"])
    assert rel(got, o * mask[..., None]) < 1e-5


def test_gelu_tanh_and_mish_formulas():
    x = torch.linspace(-6, 6, 1001)
    g = 0.5 * x * (1 + torch.tanh(math.sqrt(2 / math.pi) * (x + 0.044715 * x ** 3)))
    assert torch.allclose(F.gelu(x, approximate="tanh"), g, atol=1e-6)
    assert torch.allclose(F.mish(x), x * torch.tanh(F.softplus(x)), atol=1e-6)


def test_conv1d_nlc_is_mlx_layout_conv():
    x = torch.randn(2, 30, 32); w_mlx = torch.randn(32, 5, 8); b = torch.randn(32)     # groups=4
    got = O.conv1d_nlc(x, w_mlx, b, padding=2, groups=4)
    # direct definition
    ref = torch.zeros(2, 30, 32)
    xp = F.pad(x, (0, 0, 2, 2))
    for o in range(32):
        g = o // 8
        for k in range(5):
            ref[:, :, o] += (xp[:, k:k + 30, g * 8:(g + 1) * 8] * w_mlx[o, k]).sum(-1)
    assert torch.allclose(got, ref + b, atol=1e-4)


def test_grn_includes_padded_rows_and_matches_definition():
    x = torch.randn(2, 17, 12); gamma = torch.randn(1, 1, 12); beta = torch.randn(1, 1, 12)
    Gx = x.pow(2).sum(1, keepdim=True).sqrt()
    ref = gamma * (x * (Gx / (Gx.mean(-1, keepdim=True) + 1e-6))) + beta + x
    assert torch.allclose(O.grn(x, gamma, beta), ref, atol=1e-6)


# ---------------- solvers / schedule / prologue ----------------
@pytest.mark.parametrize("solver,order", [(O.odeint_euler, 1), (O.odeint_midpoint, 2), (O.odeint_rk4, 4)])
def test_solver_convergence_order(solver, order):
    f = lambda t, y: -y
    errs = []
    for steps in (9, 17):
        y = solver(f, torch.ones(1, dtype=torch.float64), torch.linspace(0, 1, steps, dtype=torch.float64))
        assert y.shape[0] == steps                      # all grid states are returned (cfm.py:61)
        errs.append(abs(y[-1].item() - math.exp(-1)))
    assert errs[0] / errs[1] == pytest.approx(2 ** order, rel=0.25)


def test_schedule_known_answers(golden_dir):
    z = np.load(os.path.join(golden_dir, "schedule_kat.npz"))
    for steps in (2, 8, 32):
        for sway, tag in ((None, "none"), (-1.0, "m1")):
            t = O.time_grid(steps, sway).numpy()
            np.testing.assert_allclose(t, z[f"t_{steps}_{tag}"], atol=1e-7)
            assert t.shape == (steps,) and t[0] == 0 and abs(t[-1] - 1) < 1e-6     # steps = grid POINTS
    assert O.dit_forwards_per_sample(32, "euler", 2.0) == 62
    assert O.dit_forwards_per_sample(32, "midpoint", 2.0) == 124
    assert O.dit_forwards_per_sample(8, "rk4", 2.0) == 56
    assert O.dit_forwards_per_sample(8, "rk4", 0.0) == 28


def test_sample_prologue_edge_cases():
    W = {}
    cond = torch.randn(1, 10, 100)
    # text longer than the audio: lens = max(text_len, cond_len); duration = max(lens + 1, duration)
    text = torch.randint(0, 5, (1, 14), dtype=torch.int32)
    p = O.sample_prologue(cond, text, 12, W)
    assert p.duration.tolist() == [15] and p.cond.shape == (1, 15, 100) and p.mask is None
    assert p.cond_mask[0, :, 0].sum().item() == 14
    # duration above max_duration is clipped
    p = O.sample_prologue(cond, text[:, :5], 5000, W, max_duration=64)
    assert p.duration.tolist() == [64]
    # batch > 1 gets a mask from the durations
    cond2 = torch.randn(2, 10, 100)
    text2 = torch.tensor([[1, 2, 3, -1], [1, 2, -1, -1]], dtype=torch.int32)
    p = O.sample_prologue(cond2, text2, torch.tensor([20, 16]), W)
    assert p.mask.shape == (2, 20) and p.mask.sum(-1).tolist() == [20, 16]
    with pytest.raises(ValueError):
        O.sample_prologue(cond, text, None, W)


def test_text_embedding_mask_uses_undropped_ids():
    cfg = GATE_CONFIG
    W = random_dit_weights(cfg, seed=2)
    text = torch.tensor([[5, 7, 9, -1, -1]], dtype=torch.int32)
    a = O.text_embedding(text, 8, False, W, ocfg_of(cfg))
    b = O.text_embedding(text, 8, True, W, ocfg_of(cfg))
    assert a.shape == b.shape == (1, 8, 512)
    assert (a[0, 3:] == 0).all() and (b[0, 3:] == 0).all()       # padded rows are zero in both branches
    assert b[0, :3].abs().sum() > 0 and not torch.allclose(a[0, :3], b[0, :3])


# ---------------- golden fixtures (regression pin of the oracle itself) ----------------
def test_dit_forward_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "dit_gate_forward.npz"))
    cfg = GATE_CONFIG
    W = random_dit_weights(cfg, seed=int(z["weight_seed"]))
    lens = torch.from_numpy(z["lens"]); N = z["x"].shape[1]
    mask = torch.arange(N)[None] < lens[:, None]
    out = O.dit_forward(torch.from_numpy(z["x"]), torch.from_numpy(z["cond"]), torch.from_numpy(z["text"]),
                        torch.tensor(float(z["t"])), False, False, mask, W, ocfg_of(cfg))
    assert rel(out, torch.from_numpy(z["out"])) < 2e-5


def test_sample_golden_and_bf16_drift(golden_dir):
    z = np.load(os.path.join(golden_dir, "sample_gate.npz"))
    cfg = GATE_CONFIG
    W = random_dit_weights(cfg, seed=int(z["weight_seed"]))
    args = (torch.from_numpy(z["cond"]), torch.from_numpy(z["text"]), int(z["duration"]), W, ocfg_of(cfg))
    y0 = torch.from_numpy(z["y0"])
    out, traj = O.sample(*args, steps=4, method="euler", cfg_strength=2.0, sway_sampling_coef=-1.0, y0=y0)
    assert traj.shape == (4, 1, 96, 100)
    assert rel(out, torch.from_numpy(z["euler_out"])) < 5e-5
    # the first 40 frames of `out` are the reference mel written back (cfm.py:395-397)
    assert torch.equal(out[0, :40], args[0][0])
    # derived tolerance: bf16 tensor-core operands drift ~1e-3 on this config; the GPU tests allow 3x
    out16, _ = O.sample(*args, steps=4, method="euler", cfg_strength=2.0, sway_sampling_coef=-1.0, y0=y0,
                        prec=O.Precision(True))
    drift = rel(out16, out)
    assert 1e-5 < drift < 1e-2


# ---------------- Vocos restatement ----------------
def test_istft_window_sq_trim_equals_torch_istft():
    vc = O.VocosConfig(istft_norm="window_sq", istft_trim=True)
    spec = torch.randn(20, 513, dtype=torch.complex64)
    spec[:, 0] = spec[:, 0].real + 0j; spec[:, -1] = spec[:, -1].real + 0j
    got = O.istft(spec, vc)
    ref = torch.istft(spec.T[None], n_fft=1024, hop_length=256, win_length=1024, window=torch.hann_window(1024),
                      center=True)[0]
    assert got.shape == ref.shape and torch.allclose(got, ref, atol=2e-5)


def test_vocos_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "vocos_small.npz"))
    vw = random_vocos_weights(VocosConfig(), seed=int(z["weight_seed"]))
    mel = torch.from_numpy(z["mel"])
    w1 = O.vocos_decode(mel, vw, O.VocosConfig())
    assert w1.shape == (11 * 256 + 1024,) and rel(w1, torch.from_numpy(z["wave_window"])) < 5e-5
    w2 = O.vocos_decode(mel, vw, O.VocosConfig(istft_norm="window_sq", istft_trim=True))
    assert w2.shape == (11 * 256,) and rel(w2, torch.from_numpy(z["wave_window_sq_trim"])) < 5e-5


# ---------------- DurationPredictor restatement (SURVEY §8f row 1) ----------------
def test_duration_predictor_golden_and_structure(golden_dir):
    from f5_tts_mlx_b200.weights import random_duration_weights
    z = np.load(os.path.join(golden_dir, "duration_small.npz"))
    W = {"duration." + k: v for k, v in random_duration_weights(seed=int(z["weight_seed"])).items()}
    mel, text, lens = torch.from_numpy(z["mel"]), torch.from_numpy(z["text"]), torch.from_numpy(z["lens"])
    sec = O.duration_predictor(mel, text, W, O.DurationConfig(), lens=lens)
    assert sec.shape == (2,) and (sec > 0).all()                       # Softplus output
    assert rel(sec, torch.from_numpy(z["seconds"])) < 2e-5
    # frames beyond lens[b] are zeroed on input but still attended to (no mask is passed, duration.py:245)
    mel2 = mel.clone(); mel2[1, 61:] = 123.0
    assert torch.allclose(O.duration_predictor(mel2, text, W, O.DurationConfig(), lens=lens), sec, atol=1e-6)
    # RMSNorm as used by norm_out: x * rsqrt(mean(x^2) + 1e-5) * w
    x = torch.randn(3, 7, 512)
    ref = torch.nn.functional.rms_norm(x, (512,), W["duration.transformer.norm_out.weight"], eps=1e-5)
    got = x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + 1e-5) * W["duration.transformer.norm_out.weight"]
    assert torch.allclose(got, ref, atol=1e-5)


def test_per_operator_known_answers(golden_dir):
    """SURVEY §8c item 4: per-operator input/output pairs (tiny DiT: dim 128, 2 heads, 1 block), generated by
    tests/golden/make_golden.py section (g).  Pins every building block of the oracle separately, so a regression is
    localised to the operator, not just visible in the end-to-end fixtures."""
    from f5_tts_mlx_b200.weights import DiTConfig as PkgDiTConfig
    z = np.load(os.path.join(golden_dir, "ops_small.npz"))
    tiny = PkgDiTConfig(dim=128, depth=1, heads=2, ff_mult=2, text_dim=64, conv_layers=1, text_num_embeds=50)
    tcfg = ocfg_of(tiny)
    W = random_dit_weights(tiny, seed=int(z["weight_seed"]))
    x, text, xt = torch.from_numpy(z["x"]), torch.from_numpy(z["text"]), torch.from_numpy(z["xt"])
    B, N, _ = x.shape
    mask = torch.arange(N)[None, :] < torch.tensor([40, 23])[:, None]
    rope = O.rotary_freqs(N)
    t_emb = O.timestep_embedding(torch.tensor([0.25, 0.9]), W)
    blk = "transformer.text_embed.text_blocks.layers.0."
    got = {
        "time_embed": t_emb,
        "grn": O.grn(torch.randn(B, N, 128, generator=torch.Generator().manual_seed(6)), W[blk + "grn.gamma"],
                     W[blk + "grn.beta"]),
        "convnext": O.convnext_v2_block(xt, W, blk),
        "text_embed": O.text_embedding(text, N, False, W, tcfg),
        "text_embed_drop": O.text_embedding(text, N, True, W, tcfg),
        "conv_pos": O.conv_position_embedding(x, W),
        "attention": O.attention(x, mask, rope, W, "transformer.transformer_blocks.0.attn.", 2),
        "attention_nomask": O.attention(x, None, rope, W, "transformer.transformer_blocks.0.attn.", 2),
        "dit_block": O.dit_block(x, t_emb, mask, rope, W, 0, tcfg),
        "rope_q": O.apply_rotary_pos_emb(x[:, None, :, :64], rope),
    }
    for k, v in got.items():
        assert v.shape == z[k].shape, k
        assert rel(v, torch.from_numpy(z[k])) < 2e-5, k
    # structure the fixtures must show: padded text rows are zero; masking changes only what it should
    assert (got["text_embed"][1, 7:] == 0).all() and (got["text_embed_drop"][1, 7:] == 0).all()
    assert torch.equal(got["attention"][1, 23:], torch.zeros_like(got["attention"][1, 23:]))     # x * mask (dit.py:172-173)
    assert rel(got["attention"][0], got["attention_nomask"][0]) < 1e-6                           # full-length row unaffected


# ---------------- fused AdaLN restatement + the full-size fixtures ----------------
def test_adaln_linear_linearity_identity_and_emulation():
    """oracle.adaln_linear: Linear(LN(x)(1+s)+b) == rstd * ((x(1+s)) W^T - mean * c1) + c2 exactly (float64), the fp32
    path is the reference formula, and the bf16-rounded variants (separate LN kernel / LN by linearity) drift alike."""
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 50, 256, generator=g) * 1.5 + 0.3
    s = torch.randn(2, 256, generator=g) * 0.3; b = torch.randn(2, 256, generator=g) * 0.5
    w = torch.randn(384, 256, generator=g) / 16; bias = torch.randn(384, generator=g)
    ref = F.linear(F.layer_norm(x, (256,), eps=1e-6) * (1 + s[:, None]) + b[:, None], w, bias)
    assert torch.equal(O.adaln_linear(x, s, b, w, bias), ref)
    xd, sd, bd, wd, biasd = (t.double() for t in (x, s, b, w, bias))
    mu = xd.mean(-1, keepdim=True); rstd = torch.rsqrt(xd.var(-1, unbiased=False, keepdim=True) + 1e-6)
    lin = rstd * (F.linear(xd * (1 + sd[:, None]), wd) - mu * F.linear(1 + sd, wd)[:, None]) + F.linear(bd, wd, biasd)[:, None]
    direct = F.linear((xd - mu) * rstd * (1 + sd[:, None]) + bd[:, None], wd, biasd)
    assert (lin - direct).abs().max().item() < 1e-10
    d_sep = rel(O.adaln_linear(x, s, b, w, bias, O.Precision(True, False)), ref)
    d_lin = rel(O.adaln_linear(x, s, b, w, bias, O.Precision(True, True)), ref)
    assert 0 < d_sep < 5e-3 and 0 < d_lin < 5e-3 and d_lin < 2 * d_sep


def test_full_size_golden_fixtures_present_and_inputs_reproducible(golden_dir):
    """tests/golden/full_cfg{2,3,5}_*.npz (BASELINE configs 2, 3, 5; generated by make_golden_full.py with this
    oracle): shapes, finite values, measured bf16 drift in the expected range, and the seeded inputs regenerate
    to the stored checksum on this torch build."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden_full", os.path.join(golden_dir, "make_golden_full.py"))
    G = importlib.util.module_from_spec(spec); spec.loader.exec_module(G)
    for name, fn, keys in (("full_cfg2_sample", G.inputs_cfg2, {"out": (1, 937, 100), "traj_mid": (1, 937, 100)}),
                           ("full_cfg3_sample", G.inputs_cfg3, {"out_0": (937, 100), "out_37": (937, 100)}),
                           ("full_cfg5_long", G.inputs_cfg5, {"out_sub6": (938, 100), "fwd_sub6": (938, 100)})):
        z = np.load(os.path.join(golden_dir, name + ".npz"))
        for k, shp in keys.items():
            assert z[k].shape == shp and np.isfinite(z[k]).all(), (name, k, z[k].shape)
        assert 2e-4 < float(z["drift"]) < 8e-3
        cond, text, y0, N, kw = fn()
        assert np.allclose(G.input_checksum(cond, text, y0), z["input_checksum"], rtol=1e-9), name
