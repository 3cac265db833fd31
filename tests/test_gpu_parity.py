"""-m gpu: the parity tests proper — CUDA path (through the C ABI and the reference-shaped Python
surface) vs the CPU oracle on the same seeded inputs, vs the committed golden fixtures, and
size-independent properties at the full BASELINE sizes.

Tolerance (derived, not guessed — see tests/test_oracle_pins.py::test_sample_golden_and_bf16_drift):
the oracle with bf16-rounded tensor-core operands drifts 1e-3 .. 4e-3 (rel. L2) from the fp32
oracle on these configs; the CUDA path must stay within 3x that measured drift (and an absolute
cap of 2e-2)."""
import os

import numpy as np
import pytest
import torch

from oracle import f5_oracle as O
from helpers import make_dit, ocfg_of, rel, synth_audio

pytestmark = pytest.mark.gpu
dev = "cuda"


@pytest.fixture(scope="module")
def gate():
    from f5_tts_mlx_b200.weights import GATE_CONFIG, random_dit_weights
    W = random_dit_weights(GATE_CONFIG, seed=1234)
    return GATE_CONFIG, W, make_dit(GATE_CONFIG, W)


def within_drift(got, ref_fp32, ref_bf16emu, factor=3.0, cap=2e-2):
    drift = rel(ref_bf16emu, ref_fp32)
    r = rel(got, ref_fp32)
    assert torch.isfinite(got).all()
    assert r < min(max(factor * drift, 2e-3), cap), f"rel {r:.3e} vs drift {drift:.3e}"
    return r, drift


# ---------------- DiT forward ----------------
def test_dit_forward_golden_fixture(gate, golden_dir):
    cfg, W, model = gate
    z = np.load(os.path.join(golden_dir, "dit_gate_forward.npz"))
    lens = torch.from_numpy(z["lens"]); N = z["x"].shape[1]
    mask = (torch.arange(N)[None] < lens[:, None]).to(dev)
    args = (torch.from_numpy(z["x"]).to(dev), torch.from_numpy(z["cond"]).to(dev), torch.from_numpy(z["text"]).to(dev),
            torch.tensor(float(z["t"])))
    out = model(*args, False, False, mask).cpu()
    assert rel(out, torch.from_numpy(z["out"])) < 1e-2
    out_d = model(*args, True, True, mask).cpu()
    assert rel(out_d, torch.from_numpy(z["out_drop"])) < 1e-2


@pytest.mark.parametrize("B,N,nt,drops,lens", [(1, 200, 40, (False, False), None), (1, 200, 40, (True, False), None),
                                               (1, 130, 300, (False, True), None), (2, 300, 60, (False, False), [300, 211]),
                                               (1, 5, 3, (False, False), None)])
def test_dit_forward_vs_oracle(gate, B, N, nt, drops, lens):
    cfg, W, model = gate
    g = torch.Generator().manual_seed(B * 1000 + N)
    x = torch.randn(B, N, 100, generator=g); cond = torch.randn(B, N, 100, generator=g) * 2 - 1
    text = torch.randint(0, 2545, (B, nt), generator=g, dtype=torch.int32)
    if B > 1:
        text[1, nt - 17:] = -1
    t = torch.tensor(0.37)
    mask = (torch.arange(N)[None] < torch.tensor(lens)[:, None]) if lens is not None else None
    ref = O.dit_forward(x, cond, text, t, drops[0], drops[1], mask, W, ocfg_of(cfg))
    ref16 = O.dit_forward(x, cond, text, t, drops[0], drops[1], mask, W, ocfg_of(cfg), O.Precision(True))
    got = model(x.to(dev), cond.to(dev), text.to(dev), t, drops[0], drops[1], mask.to(dev) if mask is not None else None).cpu()
    within_drift(got, ref, ref16)


# ---------------- sample(): BASELINE config 1 (the numerics gate) and the other solvers ----------------
def test_sample_config1_numerics_gate(gate):
    """BASELINE.json configs[0]: single 10 s utterance (937 frames), 4-layer/512-dim DiT random-init,
    Euler, steps=8 grid points, CFG 2, sway -1 — (out mel, trajectory[-1]) vs the CPU oracle."""
    from f5_tts_mlx_b200 import F5TTS
    cfg, W, model = gate
    g = torch.Generator().manual_seed(1)
    N, nref = 937, 328
    cond = (torch.randn(1, nref, 100, generator=g) * 2.24 - 1.27).clamp(-11.51, 5)
    text = torch.randint(0, 2545, (1, 152), generator=g, dtype=torch.int32)
    y0 = torch.randn(1, 100, N, generator=g).permute(0, 2, 1).contiguous()
    kw = dict(steps=8, method="euler", cfg_strength=2.0, sway_sampling_coef=-1.0, y0=y0)
    ref, ref_traj = O.sample(cond, text, N, W, ocfg_of(cfg), **kw)
    ref16, _ = O.sample(cond, text, N, W, ocfg_of(cfg), prec=O.Precision(True), **kw)
    f5 = F5TTS(model)
    for graph in (False, True):
        f5.use_cuda_graph = graph
        out, traj = f5.sample(cond.to(dev), text, N, **kw)
        assert traj.shape == ref_traj.shape == (8, 1, N, 100)
        r, drift = within_drift(out.cpu(), ref, ref16)
        assert rel(traj[-1].cpu(), ref_traj[-1]) < 3 * max(drift, 1e-3)
        assert (out.cpu() - ref).abs().max().item() < 5e-2               # log-mel units
        assert torch.equal(out[0, :nref].cpu(), cond[0])                  # ref frames written back (cfm.py:395-397)
    # replaying the captured graph with new noise gives the new answer, not the cached one
    y1 = torch.randn(1, 100, N, generator=g).permute(0, 2, 1).contiguous()
    out1, _ = f5.sample(cond.to(dev), text, N, **{**kw, "y0": y1})
    ref1, _ = O.sample(cond, text, N, W, ocfg_of(cfg), **{**kw, "y0": y1})
    assert rel(out1.cpu(), ref1) < 1e-2


def test_sample_golden_fixture_all_solvers(gate, golden_dir):
    from f5_tts_mlx_b200 import F5TTS
    cfg, W, model = gate
    z = np.load(os.path.join(golden_dir, "sample_gate.npz"))
    cond, text, y0, N = torch.from_numpy(z["cond"]), torch.from_numpy(z["text"]), torch.from_numpy(z["y0"]), int(z["duration"])
    f5 = F5TTS(model)
    out, traj = f5.sample(cond.to(dev), text, N, steps=4, method="euler", cfg_strength=2.0, sway_sampling_coef=-1.0, y0=y0)
    assert rel(out.cpu(), torch.from_numpy(z["euler_out"])) < 1e-2
    assert rel(traj[-1].cpu(), torch.from_numpy(z["euler_traj_last"])) < 1e-2
    out, _ = f5.sample(cond.to(dev), text, N, steps=3, method="midpoint", cfg_strength=0.0, sway_sampling_coef=None, y0=y0)
    assert rel(out.cpu(), torch.from_numpy(z["midpoint_nocfg_out"])) < 1e-2
    out, _ = f5.sample(cond.to(dev), text, N, steps=3, method="rk4", cfg_strength=2.0, sway_sampling_coef=-1.0, y0=y0)
    assert rel(out.cpu(), torch.from_numpy(z["rk4_out"])) < 1e-2


def test_sample_ragged_batch_and_text_longer_than_audio(gate):
    """batch > 1 => key-padding mask + zeroed padded query rows (dit.py:161-173), per-utterance
    durations, lens = max(text_len, cond_len) (cfm.py:301-303)."""
    from f5_tts_mlx_b200 import F5TTS
    cfg, W, model = gate
    g = torch.Generator().manual_seed(5)
    cond = (torch.randn(2, 50, 100, generator=g) * 2.24 - 1.27)
    text = torch.randint(0, 2545, (2, 60), generator=g, dtype=torch.int32); text[1, 20:] = -1
    dur = torch.tensor([120, 90])
    y0 = torch.randn(2, 120, 100, generator=g); y0[1, 90:] = 0
    kw = dict(steps=3, method="midpoint", cfg_strength=2.0, sway_sampling_coef=-1.0, y0=y0)
    ref, _ = O.sample(cond, text, dur, W, ocfg_of(cfg), **kw)
    ref16, _ = O.sample(cond, text, dur, W, ocfg_of(cfg), prec=O.Precision(True), **kw)
    out, traj = F5TTS(model).sample(cond.to(dev), text, dur, **kw)
    assert out.shape == ref.shape == (2, 120, 100)
    within_drift(out.cpu(), ref, ref16)


def test_sample_seeded_noise_is_deterministic_and_same_per_element(gate):
    from f5_tts_mlx_b200 import F5TTS
    cfg, W, model = gate
    cond = torch.randn(2, 30, 100).to(dev)
    text = torch.randint(0, 100, (2, 10), dtype=torch.int32)
    f5 = F5TTS(model)
    a, ta = f5.sample(cond, text, 64, steps=2, method="euler", seed=3)
    b, tb = f5.sample(cond, text, 64, steps=2, method="euler", seed=3)
    assert torch.equal(a, b)
    assert torch.equal(ta[0, 0], ta[0, 1])            # same seed re-applied per element (cfm.py:371-373)


# ---------------- full-size properties: BASELINE configs 2-3 shapes on the base model ----------------
@pytest.fixture(scope="module")
def base():
    from f5_tts_mlx_b200.weights import BASE_CONFIG, random_dit_weights
    W = random_dit_weights(BASE_CONFIG, seed=1234)
    return BASE_CONFIG, W, make_dit(BASE_CONFIG, W)


def test_base_model_single_forward_vs_oracle(base):
    """One full-size DiT evaluation (22 layers, 1024-dim, N = 937) against the oracle (a few CPU seconds)."""
    cfg, W, model = base
    g = torch.Generator().manual_seed(2)
    N = 937
    x = torch.randn(1, N, 100, generator=g); cond = (torch.randn(1, N, 100, generator=g) * 2.24 - 1.27); cond[:, 328:] = 0
    text = torch.randint(0, 2545, (1, 152), generator=g, dtype=torch.int32)
    t = torch.tensor(0.25)
    ref = O.dit_forward(x, cond, text, t, False, False, None, W, ocfg_of(cfg))
    ref16 = O.dit_forward(x, cond, text, t, False, False, None, W, ocfg_of(cfg), O.Precision(True))
    got = model(x.to(dev), cond.to(dev), text.to(dev), t).cpu()
    within_drift(got, ref, ref16)


def test_base_model_batched_cfg_equals_two_unbatched_passes_and_batch_invariance(base):
    """Properties that need no oracle at full size: (1) the doubled-batch CFG step equals
    pred + (pred - null) * cfg from two separate forwards (cfm.py:342-364); (2) an utterance gives
    the same result alone and inside a batch of identical utterances (no cross-utterance coupling)."""
    from f5_tts_mlx_b200 import F5TTS
    cfg, W, model = base
    g = torch.Generator().manual_seed(3)
    N, nref = 937, 328
    cond = (torch.randn(1, nref, 100, generator=g) * 2.24 - 1.27).clamp(-11.51, 5).to(dev)
    text = torch.randint(0, 2545, (1, 152), generator=g, dtype=torch.int32)
    y0 = torch.randn(1, N, 100, generator=g).to(dev)
    f5 = F5TTS(model)
    out, traj = f5.sample(cond, text, N, steps=2, method="euler", cfg_strength=2.0, sway_sampling_coef=None, y0=y0)
    step_cond = torch.zeros(1, N, 100, device=dev); step_cond[:, :nref] = cond
    t0 = torch.tensor(0.0)
    pred = model(y0, step_cond, text.to(dev), t0, False, False)
    null = model(y0, step_cond, text.to(dev), t0, True, True)
    y1 = y0 + 1.0 * (pred + (pred - null) * 2.0)
    assert rel(traj[-1], y1) < 1e-5
    cond3, text3, y03 = cond.repeat(3, 1, 1), text.repeat(3, 1), y0.repeat(3, 1, 1)
    out3, _ = f5.sample(cond3, text3, N, steps=2, method="euler", cfg_strength=2.0, sway_sampling_coef=None, y0=y03)
    assert rel(out3[1], out[0]) < 1e-5 and torch.equal(out3[0], out3[2])


def test_base_model_long_form_60s_runs_and_is_finite(base):
    """BASELINE configs[4] shape: N = 5625 frames (60 s), max_duration passed explicitly; text positions
    beyond 4095 reuse the last table row (rope.py:83)."""
    from f5_tts_mlx_b200 import F5TTS
    cfg, W, model = base
    g = torch.Generator().manual_seed(4)
    cond = (torch.randn(1, 499, 100, generator=g) * 2.24 - 1.27).to(dev)
    text = torch.randint(0, 2545, (1, 900), generator=g, dtype=torch.int32)
    out, traj = F5TTS(model).sample(cond, text, 5625, steps=3, method="euler", cfg_strength=2.0, seed=0, max_duration=8192,
                                    return_trajectory=False)
    assert out.shape == (1, 5625, 100) and torch.isfinite(out).all()
    capped, _ = F5TTS(model).sample(cond, text, 5625, steps=2, method="euler", cfg_strength=0.0, seed=0, return_trajectory=False)
    assert capped.shape == (1, 4096, 100)             # default max_duration = 4096 (cfm.py:277,318)


# ---------------- audio front-end / vocoder ----------------
def test_mel_golden_fixture_and_oracle(golden_dir):
    from f5_tts_mlx_b200 import MelSpec
    z = np.load(os.path.join(golden_dir, "mel_fixture.npz"))
    x = torch.from_numpy(z["pcm"].astype(np.float32) / 32768.0)
    got = MelSpec()(x.to(dev)).cpu()[0]
    assert got.shape == (93, 100) and (got - torch.from_numpy(z["mel"])).abs().max().item() < 2e-3
    for L in (240000, 127985, 1024, 700, 256):
        a = synth_audio(L, seed=L)
        got, ref = MelSpec()(a.to(dev)).cpu(), O.log_mel_spectrogram(a)
        assert got.shape == ref.shape == (1, L // 256, 100)
        assert (got - ref).abs().max().item() < 3e-3
    xb = torch.stack([synth_audio(24000, 1), synth_audio(24000, 2)])
    assert (MelSpec()(xb.to(dev)).cpu() - O.log_mel_spectrogram(xb)).abs().max().item() < 3e-3


@pytest.mark.parametrize("norm,trim", [("window", False), ("window_sq", True)])
def test_vocos_vs_oracle_and_golden(golden_dir, norm, trim):
    from f5_tts_mlx_b200.vocos import Vocos
    from f5_tts_mlx_b200.weights import VocosConfig, random_vocos_weights
    vc, ovc = VocosConfig(istft_norm=norm, istft_trim=trim), O.VocosConfig(istft_norm=norm, istft_trim=trim)
    vw = random_vocos_weights(vc, seed=4321)
    voc = Vocos(vc, dev).load_weights(vw)
    z = np.load(os.path.join(golden_dir, "vocos_small.npz"))
    got = voc.decode(torch.from_numpy(z["mel"]).to(dev)).cpu()
    gold = torch.from_numpy(z["wave_window" if norm == "window" else "wave_window_sq_trim"])
    assert got.shape == gold.shape and rel(got, gold) < 2e-2
    for n in (2, 499, 937):
        mel = (torch.randn(1, n, 100) * 2.24 - 1.27).clamp(-11.5, 5)
        ref, ref16 = O.vocos_decode(mel, vw, ovc), O.vocos_decode(mel, vw, ovc, O.Precision(True))
        got = voc.decode(mel.to(dev)).cpu()
        assert got.shape == ref.shape
        within_drift(got, ref, ref16)
        snr = 10 * torch.log10(ref.pow(2).sum() / (got - ref).pow(2).sum()).item()
        assert snr > 40.0, f"SNR {snr:.1f} dB"


def test_end_to_end_raw_wave_to_waveform(gate):
    """sample(raw wave, text) with a vocoder: mel front-end -> ODE -> Vocos, output is a 1-D wave whose
    first len(audio) samples are the re-synthesised reference (generate.py:183 strips them)."""
    from f5_tts_mlx_b200 import F5TTS
    from f5_tts_mlx_b200.vocos import Vocos
    from f5_tts_mlx_b200.weights import VocosConfig, random_vocos_weights
    cfg, W, model = gate
    vw = random_vocos_weights()
    voc = Vocos(VocosConfig(), dev).load_weights(vw)
    audio = synth_audio(256 * 80, 9)
    text = torch.randint(0, 2545, (1, 30), dtype=torch.int32)
    N = 200
    y0 = torch.randn(1, N, 100)
    kw = dict(steps=3, method="euler", cfg_strength=2.0, sway_sampling_coef=-1.0, y0=y0)
    wave, traj = F5TTS(model, vocoder=voc.decode).sample(audio[None].to(dev), text, N, **kw)
    ref, _ = O.sample(audio[None], text, N, W, ocfg_of(cfg), vocoder=lambda m: O.vocos_decode(m, vw), **kw)
    assert wave.ndim == 1 and wave.shape == ref.shape == ((N - 1) * 256 + 1024,)
    assert rel(wave.cpu(), ref) < 3e-2


# ---------------- DurationPredictor (SURVEY §8f row 1) ----------------
def test_duration_predictor_vs_oracle_and_golden(golden_dir):
    from f5_tts_mlx_b200.duration import DurationPredictor, DurationTransformer
    from f5_tts_mlx_b200.weights import random_duration_weights
    z = np.load(os.path.join(golden_dir, "duration_small.npz"))
    dW = random_duration_weights(seed=int(z["weight_seed"]))
    dWo = {"duration." + k: v for k, v in dW.items()}
    pred = DurationPredictor(DurationTransformer(dim=512, depth=8, heads=8, text_dim=512, ff_mult=2, conv_layers=2,
                                                 text_num_embeds=2545), device=dev).load_weights(dW)
    mel, text, lens = torch.from_numpy(z["mel"]), torch.from_numpy(z["text"]), torch.from_numpy(z["lens"])
    got = pred(mel.to(dev), text, lens=lens).cpu()
    assert rel(got, torch.from_numpy(z["seconds"])) < 2e-2
    # text longer than the mel (the mel is padded to the text length, duration.py:220-222), batch 1, no lens
    g = torch.Generator().manual_seed(8)
    mel1 = torch.randn(1, 40, 100, generator=g); text1 = torch.randint(0, 2545, (1, 70), generator=g, dtype=torch.int32)
    ref = O.duration_predictor(mel1, text1, dWo, O.DurationConfig())
    ref16 = O.duration_predictor(mel1, text1, dWo, O.DurationConfig(), prec=O.Precision(True))
    got1 = pred(mel1.to(dev), text1).cpu()
    assert abs(got1.item() - ref.item()) < max(3 * abs(ref16.item() - ref.item()), 2e-2 * abs(ref.item()))


def test_sample_with_duration_predictor(gate):
    """duration=None routes through predict_duration (cfm.py:253-262, integer frame rate 93)."""
    from f5_tts_mlx_b200 import F5TTS
    from f5_tts_mlx_b200.duration import DurationPredictor, DurationTransformer
    from f5_tts_mlx_b200.weights import random_duration_weights
    cfg, W, model = gate
    dW = random_duration_weights(seed=5)
    pred = DurationPredictor(DurationTransformer(dim=512, depth=8, heads=8, text_dim=512, ff_mult=2, conv_layers=2,
                                                 text_num_embeds=2545), device=dev).load_weights(dW)
    g = torch.Generator().manual_seed(9)
    cond = (torch.randn(1, 60, 100, generator=g) * 2.24 - 1.27)
    text = torch.randint(0, 2545, (1, 25), generator=g, dtype=torch.int32)
    secs = O.duration_predictor(cond, text, {"duration." + k: v for k, v in dW.items()}, O.DurationConfig()).item()
    expect = max(60 + 1, int(secs * 93 / 1.0))
    out, _ = F5TTS(model, duration_predictor=pred).sample(cond.to(dev), text, None, steps=2, method="euler", seed=1)
    assert abs(out.shape[1] - expect) <= 1 and torch.isfinite(out).all()
    with pytest.raises(ValueError):
        F5TTS(model).sample(cond.to(dev), text, None, steps=2, method="euler")


def test_generate_end_to_end_serial_and_batched_sentences(tmp_path):
    """generate.py:113-244 through the package's own `generate()`: wav in -> wav out on the base architecture
    (random weights), serial per-sentence loop (the reference's) and the one-ragged-batch extension.  Checks
    the bookkeeping the reference does around sample(): RMS normalisation, sentence split, estimated duration,
    reference-audio stripping, concatenation, 16-bit wav writing."""
    from f5_tts_mlx_b200 import F5TTS
    from f5_tts_mlx_b200 import generate as G
    torch.manual_seed(0)
    ref = 0.02 * torch.randn(2 * 24000)                                      # quiet clip -> exercises the RMS branch
    G.write_wav(str(tmp_path / "ref.wav"), ref)
    text, ref_text = "Hello there. This is a test!", "some reference text."
    n_ref = ref.shape[0]
    expect = 0
    f5 = F5TTS.from_pretrained("random")
    for s in G.split_sentences(text):
        frames = int(G.estimated_duration(ref, ref_text, s) * G.FRAMES_PER_SEC)
        frames = max(frames, n_ref // 256 + 1)
        expect += f5._vocoder.__self__.out_len(frames) - n_ref          # un-trimmed ISTFT: (frames-1)*256 + 1024
    waves = {}
    for batched in (False, True):
        out = tmp_path / f"out{int(batched)}.wav"
        w = G.generate(text, estimate_duration=True, ref_audio_path=str(tmp_path / "ref.wav"), ref_audio_text=ref_text,
                       steps=4, method="euler", seed=7, output_path=str(out), f5tts=f5, batch_sentences=batched)
        assert w.ndim == 1 and torch.isfinite(w).all() and float(w.abs().max()) > 0
        assert abs(w.shape[0] - expect) <= 3 * 256, (w.shape, expect)
        back, sr = G.read_wav(str(out))
        assert sr == 24000 and back.shape[0] == w.shape[0]
        waves[batched] = w
    assert waves[False].shape == waves[True].shape
    # numerically: two sentences of the same length form an equal-length batch, so the one-batch run has no padding
    # and must reproduce the serial loop (same seed => same noise per sentence, cfm.py:371-373)
    same = "Same words here. Same words here."
    ws = [G.generate(same, estimate_duration=True, ref_audio_path=str(tmp_path / "ref.wav"), ref_audio_text=ref_text,
                     steps=4, method="euler", seed=7, f5tts=f5, batch_sentences=b) for b in (False, True)]
    assert ws[0].shape == ws[1].shape and rel(ws[1], ws[0]) < 5e-3, rel(ws[1], ws[0])
    # the serial loop's sentences shared ONE bucketed plan (frame_bucket=128): no re-capture per sentence length
    n_bucketed = sum(1 for k in f5._plans if k[-1])
    assert n_bucketed >= 1 and all(k[1] % 128 == 0 for k in f5._plans if k[-1])
    with pytest.raises(ValueError):                                           # generate.py:147-148
        import wave as wavmod
        with wavmod.open(str(tmp_path / "bad.wav"), "wb") as f:
            f.setnchannels(1); f.setsampwidth(2); f.setframerate(16000); f.writeframes(b"\0\0" * 100)
        G.generate(text, duration=3.0, ref_audio_path=str(tmp_path / "bad.wav"), f5tts=f5)
    with pytest.raises(ValueError):                                           # no duration, no estimate, no predictor
        G.generate(text, ref_audio_path=str(tmp_path / "ref.wav"), f5tts=f5)


# ---------------- multi-GPU: sharded == unsharded (needs 2 GPUs; skipped on a 1-GPU box) ----------------
def test_nccl_sharded_ragged_batch_equals_unsharded():
    """SURVEY §8e: utterances shard across ranks with ONE NCCL weight broadcast and no per-step collective; a ragged
    batch sharded over 2 GPUs (each shard padded to the global frame count) reproduces the unsharded batch."""
    import json, subprocess, sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29731",
                        os.path.join(root, "tests", "gpu_checks", "nccl_shard_check.py")],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("NCCL_SHARD_CHECK ")][-1]
    res = json.loads(line[len("NCCL_SHARD_CHECK "):])
    assert res["utterances"] == 5 and res["max_rel"] < 1e-5, res


# ---------------- full-size golden fixtures on the configurations the metric is quoted on ----------------
# tests/golden/make_golden_full.py (CPU oracle, offline): fp32 output + the measured drift of the oracle's
# bf16-operand emulation; the CUDA path must stay within 3x that drift (cap 2e-2), like everywhere else.
def _golden_full():
    import importlib.util
    p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_golden_full.py")
    spec = importlib.util.spec_from_file_location("make_golden_full", p)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _tol(drift):
    return min(max(3.0 * float(drift), 2e-3), 2e-2)


def test_full_config2_sample_32_euler_steps_vs_golden(base, golden_dir):
    """BASELINE configs[1] end to end: base model, 937 frames, Euler, 32 grid points (62 DiT evaluations), CFG 2,
    sway -1 — the whole integrated trajectory against the fp32 oracle (generated frames, and the state at grid
    point 16), through the CUDA graph the bench replays."""
    from f5_tts_mlx_b200 import F5TTS
    G = _golden_full()
    z = np.load(os.path.join(golden_dir, "full_cfg2_sample.npz"))
    cfg, W, model = base
    cond, text, y0, N, kw = G.inputs_cfg2()
    out, traj = F5TTS(model).sample(cond.to(dev), text, N, y0=y0, **kw)
    gold = torch.from_numpy(z["out"])
    nref = G.NREF10S
    r = rel(out[:, nref:].cpu(), gold[:, nref:])
    assert torch.equal(out[0, :nref].cpu(), cond[0])
    assert r < _tol(z["drift"]), f"rel {r:.3e} vs oracle bf16 drift {float(z['drift']):.3e}"
    rm = rel(traj[16].cpu(), torch.from_numpy(z["traj_mid"]))
    assert rm < _tol(z["traj_drift"][2]), f"trajectory[16] rel {rm:.3e}"
    assert (out.cpu() - gold).abs().max().item() < 0.15            # log-mel units, after 31 integration steps


def test_full_config3_batch64_midpoint_vs_golden(base, golden_dir):
    """BASELINE configs[2]: 64 equal-length utterances, midpoint, 32 grid points, CFG 2, sway -1, ONE batched sample();
    utterances 0 and 37 against the oracle run on each of them alone (utterances are independent, cfm.py:340-365)."""
    from f5_tts_mlx_b200 import F5TTS
    G = _golden_full()
    z = np.load(os.path.join(golden_dir, "full_cfg3_sample.npz"))
    cfg, W, model = base
    cond, text, y0, N, kw = G.inputs_cfg3()
    f5 = F5TTS(model)
    f5.use_cuda_graph = False            # one pass is enough here; the graph path is covered by the other tests
    out, _ = f5.sample(cond.to(dev), text, N, y0=y0, return_trajectory=False, **kw)
    assert out.shape == (G.CFG3_BATCH, N, 100)
    for u in z["checked"].tolist():
        r = rel(out[u, G.NREF10S:].cpu(), torch.from_numpy(z[f"out_{u}"])[G.NREF10S:])
        assert r < _tol(z["drift"]), f"utterance {u}: rel {r:.3e} vs drift {float(z['drift']):.3e}"
    del f5, out
    torch.cuda.empty_cache()


def test_full_config5_long_form_vs_golden(base, golden_dir):
    """BASELINE configs[4] shape: N = 5625 frames (60 s), 900 text tokens, max_duration passed explicitly
    (cfm.py:277,318): a 3-grid-point CFG sample and one forward at t = 0.25 against the oracle (every sixth frame is
    stored)."""
    from f5_tts_mlx_b200 import F5TTS
    G = _golden_full()
    z = np.load(os.path.join(golden_dir, "full_cfg5_long.npz"))
    cfg, W, model = base
    cond, text, y0, N, kw = G.inputs_cfg5()
    out, _ = F5TTS(model).sample(cond.to(dev), text, N, y0=y0, return_trajectory=False, **kw)
    assert out.shape == (1, N, 100)
    sub = out[0, ::6].cpu()
    gold = torch.from_numpy(z["out_sub6"])
    gen = torch.arange(0, N, 6) >= G.NREF60S
    r = rel(sub[gen], gold[gen])
    assert r < _tol(z["drift"]), f"rel {r:.3e} vs drift {float(z['drift']):.3e}"
    step_cond = torch.zeros(1, N, 100); step_cond[:, :G.NREF60S] = cond
    v = model(y0.to(dev), step_cond.to(dev), text.to(dev), torch.tensor(0.25)).cpu()
    rf = rel(v[0, ::6], torch.from_numpy(z["fwd_sub6"]))
    assert rf < _tol(z["fwd_drift"]), f"forward rel {rf:.3e} vs drift {float(z['fwd_drift']):.3e}"
    torch.cuda.empty_cache()


def test_fused_adaln_matches_separate_layernorm_kernels(base):
    """The AdaLN LayerNorm+modulate folded into the GEMM epilogues (default) against the same model run with the
    separate f5_ln_modulate launches: both are bf16-operand paths with different rounding points, so they agree to the
    bf16 drift level, and both stay within tolerance of the fp32 oracle (test_base_model_single_forward_vs_oracle)."""
    cfg, W, model = base
    sep = make_dit(cfg, W, fused_adaln=False)
    g = torch.Generator().manual_seed(12)
    N = 937
    x = torch.randn(1, N, 100, generator=g); cond = (torch.randn(1, N, 100, generator=g) * 2.24 - 1.27); cond[:, 328:] = 0
    text = torch.randint(0, 2545, (1, 152), generator=g, dtype=torch.int32)
    t = torch.tensor(0.6)
    a = model(x.to(dev), cond.to(dev), text.to(dev), t)
    b = sep(x.to(dev), cond.to(dev), text.to(dev), t)
    ref = O.dit_forward(x, cond, text, t, False, False, None, W, ocfg_of(cfg))
    ra, rb = rel(a.cpu(), ref), rel(b.cpu(), ref)
    assert ra < 2e-2 and rb < 2e-2 and ra < 2.0 * rb + 1e-3, (ra, rb)
    assert rel(a, b) < 2e-2
    del sep
    torch.cuda.empty_cache()



def test_frame_bucketing_one_plan_for_many_lengths_same_results(gate):
    """F5TTS.frame_bucket: utterances of 150, 201 and 255 frames share the 256-frame plan (one set of buffers, one
    captured CUDA graph) and give the results of their exact-shape plans — bucket rows are kept zero where the
    reference's zero padding is visible (conv position embedding) and masked as attention keys."""
    from f5_tts_mlx_b200 import F5TTS
    cfg, W, model = gate
    g = torch.Generator().manual_seed(21)
    cond = (torch.randn(1, 60, 100, generator=g) * 2.24 - 1.27).to(dev)
    kw = dict(steps=4, method="euler", cfg_strength=2.0, sway_sampling_coef=-1.0)
    exact, bucketed = F5TTS(model), F5TTS(model)
    bucketed.frame_bucket = 128
    plans = set()
    for N, nt in ((150, 20), (201, 31), (255, 27)):
        text = torch.randint(0, 2545, (1, nt), generator=g, dtype=torch.int32)
        y0 = torch.randn(1, N, 100, generator=g)
        a, ta = exact.sample(cond, text, N, y0=y0, **kw)
        b, tb = bucketed.sample(cond, text, N, y0=y0, **kw)
        plans.add(id(bucketed.last_plan))
        assert b.shape == a.shape == (1, N, 100) and tb.shape == ta.shape
        assert rel(b, a) < 1e-3, (N, rel(b, a))
        ref, _ = O.sample(cond.cpu(), text, N, W, ocfg_of(cfg), y0=y0, **kw)
        assert rel(b.cpu(), ref) < 1e-2
    assert len(plans) == 1 and bucketed.last_plan.session.frames == 256


def test_fp8_mode_forward_within_derived_drift(base):
    """DiT(fp8=True): the four GEMMs of every block on e4m3 operands (weights quantised per tensor at pack time,
    activations written as e4m3 by the producing kernels) — the B200 analogue of the reference's lossy `--q`
    checkpoints.  Same rule as everywhere: within 3x the drift of the oracle's emulation of exactly these rounding
    points (Precision(fp8=True)), which is ~7x the bf16 drift."""
    cfg, W, model = base
    m8 = make_dit_fp8(cfg, W)
    g = torch.Generator().manual_seed(2)
    N = 937
    x = torch.randn(1, N, 100, generator=g); cond = (torch.randn(1, N, 100, generator=g) * 2.24 - 1.27); cond[:, 328:] = 0
    text = torch.randint(0, 2545, (1, 152), generator=g, dtype=torch.int32)
    t = torch.tensor(0.25)
    ref = O.dit_forward(x, cond, text, t, False, False, None, W, ocfg_of(cfg))
    ref8 = O.dit_forward(x, cond, text, t, False, False, None, W, ocfg_of(cfg), O.Precision(True, True, True))
    got = m8(x.to(dev), cond.to(dev), text.to(dev), t).cpu()
    drift = rel(ref8, ref)
    r = rel(got, ref)
    assert 5e-3 < drift < 5e-2 and r < min(3 * drift, 1e-1), (r, drift)
    assert rel(got, ref8) < 2.0 * drift                     # and close to the emulation itself
    # through the integrator (8 Euler grid points, CFG): the e4m3 noise does not blow up
    from f5_tts_mlx_b200 import F5TTS
    nref = 328
    kw = dict(steps=8, method="euler", cfg_strength=2.0, sway_sampling_coef=-1.0, y0=x)
    out, _ = F5TTS(m8).sample(cond[:, :nref].to(dev), text, N, **kw)
    out16, _ = F5TTS(model).sample(cond[:, :nref].to(dev), text, N, **kw)
    assert torch.isfinite(out).all() and rel(out[:, nref:], out16[:, nref:]) < 1e-1
    del m8
    torch.cuda.empty_cache()


def make_dit_fp8(cfg, W):
    from f5_tts_mlx_b200 import DiT
    return DiT(dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, ff_mult=cfg.ff_mult, mel_dim=cfg.mel_dim,
               text_num_embeds=cfg.text_num_embeds, text_dim=cfg.text_dim, conv_layers=cfg.conv_layers,
               device=dev, fp8=True).load_weights(W)
