"""Records a second, independent run of the REFERENCE'S OWN CODE (needs a checkout of the reference project where
tests/mlx_shim looks for it) into ref_recomputed.npz.

make_ref_golden.py writes the ref_*.npz fixtures the oracle and the CUDA path are pinned to.  This script runs the
unmodified reference again on the shim, the way a user calls it (a fresh DiT, F5TTS.sample, log_mel_spectrogram), and
stores what it returns.  tests/test_ref_pins.py checks that the fixtures agree with this recording, so the suite
needs neither the reference nor MLX to know that the committed fixtures are what the reference computes.

    python tests/golden/make_ref_recomputed.py      # rewrites tests/golden/ref_recomputed.npz
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import mlx_shim as shim                                                  # noqa: E402
from f5_tts_mlx_b200.weights import GATE_CONFIG, random_dit_weights     # noqa: E402

torch.set_num_threads(8)
ref = shim.import_reference()
A = ref.mx.array
cfg = GATE_CONFIG
W = random_dit_weights(cfg, seed=1234)
dit = ref.dit.DiT(dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, ff_mult=cfg.ff_mult, mel_dim=cfg.mel_dim,
                  text_num_embeds=cfg.text_num_embeds, text_dim=cfg.text_dim, conv_layers=cfg.conv_layers)
dit.load_weights([(k[len("transformer."):], A(v)) for k, v in W.items()])

z = np.load(os.path.join(HERE, "ref_dit_gate.npz"))
out = dit(x=A(z["x"]), cond=A(z["cond"]), text=A(z["text"]), time=A(z["t"]), drop_audio_cond=False, drop_text=False)
# dit.py:162: mx.array has no .expand, so a batch > 1 with a key-padding mask cannot run upstream
try:
    dit(x=A(z["x2"]), cond=A(z["cond2"]), text=A(z["text2"]), time=A(z["t"]), drop_audio_cond=False, drop_text=False,
        mask=A(np.ones(z["x2"].shape[:2], dtype=bool)))
    masked_batch_error = ""
except Exception as e:                                                   # recorded, not asserted, here
    masked_batch_error = type(e).__name__

zs = np.load(os.path.join(HERE, "ref_sample_gate.npz"))
o, _ = ref.cfm.F5TTS(transformer=dit).sample(A(zs["cond"]), A(zs["text"]), int(zs["duration"]), steps=3,
                                             method="midpoint", cfg_strength=0.0, sway_sampling_coef=None, seed=7)
pcm = np.load(os.path.join(HERE, "mel_fixture.npz"))["pcm"]
mel = ref.audio.log_mel_spectrogram(A(pcm.astype(np.float32) / 32768.0))

np.savez_compressed(os.path.join(HERE, "ref_recomputed.npz"), dit_out=np.asarray(out),
                    masked_batch_error=np.array(masked_batch_error), sample_midpoint_nocfg_out=np.asarray(o),
                    mel=np.asarray(mel), weight_seed=1234)
print("masked batch:", masked_batch_error or "ran", "| size", os.path.getsize(os.path.join(HERE, "ref_recomputed.npz")))
