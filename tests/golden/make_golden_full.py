"""Full-size golden fixtures on the configurations the metric is quoted on (BASELINE.json configs 2, 3, 5),
generated offline by the CPU oracle (oracle/f5_oracle.py, pinned to the reference's own code by
tests/test_ref_pins.py).  Run in the build container (about 10 CPU-minutes on 8 cores); the GPU box only
reads the committed .npz files.

    python tests/golden/make_golden_full.py [cfg2] [cfg3] [cfg5]

Every fixture holds the fp32 oracle output and `drift` = rel-L2 distance of the oracle run with
bf16-rounded tensor-core operands (the CUDA path's precision model) from the fp32 run — the measured
quantity the GPU tolerance is derived from (CUDA must stay within 3x drift).

Inputs are NOT stored: they are regenerated from the seeds below by `inputs_cfg*()` (torch CPU
generators, same torch build on both machines), which the GPU tests import from here.
"""
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N10S, NREF10S, NTEXT = 937, 328, 152          # SURVEY §8d synthetic 10 s utterance
CFG3_BATCH, CFG3_CHECKED = 64, (0, 37)        # config 3: 64 equal-length utterances; oracle on two of them
N60S, NREF60S, NTEXT60S = 5625, 499, 900      # config 5: 60 s, text longer than... positions clamp at 4095 is exercised by N > 4096


def _cond(g, b, nref):
    return (torch.randn(b, nref, 100, generator=g) * 2.24 - 1.27).clamp(-11.51, 5.0)


def inputs_cfg2():
    g = torch.Generator().manual_seed(20202)
    cond = _cond(g, 1, NREF10S)
    text = torch.randint(0, 2545, (1, NTEXT), generator=g, dtype=torch.int32)
    y0 = torch.randn(1, 100, N10S, generator=g).permute(0, 2, 1).contiguous()
    kw = dict(steps=32, method="euler", cfg_strength=2.0, sway_sampling_coef=-1.0)
    return cond, text, y0, N10S, kw


def inputs_cfg3():
    g = torch.Generator().manual_seed(30303)
    cond = _cond(g, CFG3_BATCH, NREF10S)
    text = torch.randint(0, 2545, (CFG3_BATCH, NTEXT), generator=g, dtype=torch.int32)
    y0 = torch.randn(CFG3_BATCH, 100, N10S, generator=g).permute(0, 2, 1).contiguous()
    kw = dict(steps=32, method="midpoint", cfg_strength=2.0, sway_sampling_coef=-1.0)
    return cond, text, y0, N10S, kw


def inputs_cfg5():
    g = torch.Generator().manual_seed(50505)
    cond = _cond(g, 1, NREF60S)
    text = torch.randint(0, 2545, (1, NTEXT60S), generator=g, dtype=torch.int32)
    y0 = torch.randn(1, 100, N60S, generator=g).permute(0, 2, 1).contiguous()
    kw = dict(steps=3, method="euler", cfg_strength=2.0, sway_sampling_coef=-1.0, max_duration=8192)
    return cond, text, y0, N60S, kw


def input_checksum(cond, text, y0) -> np.ndarray:
    """Stored in every fixture: guards the GPU tests against a torch build whose CPU generator yields other inputs."""
    return np.array([cond.double().abs().sum().item(), float(text.long().sum().item()), y0.double().abs().sum().item()])


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm()).item()


def main():
    from oracle import f5_oracle as O
    from f5_tts_mlx_b200.weights import BASE_CONFIG, random_dit_weights
    torch.set_num_threads(os.cpu_count() or 8)
    which = set(sys.argv[1:]) or {"cfg2", "cfg3", "cfg5"}
    cfg = BASE_CONFIG
    W = random_dit_weights(cfg, seed=1234)
    ocfg = O.DiTConfig(dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, ff_mult=cfg.ff_mult,
                       text_num_embeds=cfg.text_num_embeds, text_dim=cfg.text_dim, conv_layers=cfg.conv_layers)
    emu = O.Precision(True)

    if "cfg2" in which:
        cond, text, y0, N, kw = inputs_cfg2()
        t0 = time.time()
        with torch.no_grad():
            out, traj = O.sample(cond, text, N, W, ocfg, y0=y0, **kw)
            out16, traj16 = O.sample(cond, text, N, W, ocfg, y0=y0, prec=emu, **kw)
        drift = _rel(out16[:, NREF10S:], out[:, NREF10S:])
        # drift of the trajectory at a few grid points: how bf16 rounding accumulates through the integrator
        marks = [1, 8, 16, 24, 31]
        tdrift = [_rel(traj16[i], traj[i]) for i in marks]
        np.savez_compressed(os.path.join(HERE, "full_cfg2_sample.npz"), out=out.numpy(), traj_mid=traj[16].numpy(),
                            drift=np.float64(drift), traj_marks=np.array(marks), traj_drift=np.array(tdrift),
                            weight_seed=1234, input_seed=20202, input_checksum=input_checksum(cond, text, y0))
        print(f"cfg2: {time.time() - t0:.0f}s drift(gen frames)={drift:.3e} traj drift {tdrift}", flush=True)

    if "cfg3" in which:
        cond, text, y0, N, kw = inputs_cfg3()
        outs, drifts = {}, {}
        t0 = time.time()
        for j, u in enumerate(CFG3_CHECKED):
            # utterances of an equal-length batch are independent (cfm.py:340-365; the batch mask is all-true):
            # the B = 1 oracle run of utterance u IS the reference result of row u of the batch
            with torch.no_grad():
                o, _ = O.sample(cond[u:u + 1], text[u:u + 1], N, W, ocfg, y0=y0[u:u + 1], **kw)
                outs[f"out_{u}"] = o[0].numpy()
                if j == 0:
                    o16, _ = O.sample(cond[u:u + 1], text[u:u + 1], N, W, ocfg, y0=y0[u:u + 1], prec=emu, **kw)
                    drifts["drift"] = np.float64(_rel(o16[:, NREF10S:], o[:, NREF10S:]))
            print(f"cfg3 utt {u}: {time.time() - t0:.0f}s", flush=True)
        np.savez_compressed(os.path.join(HERE, "full_cfg3_sample.npz"), checked=np.array(CFG3_CHECKED), weight_seed=1234,
                            input_seed=30303, input_checksum=input_checksum(cond, text, y0), **outs, **drifts)
        print("cfg3 drift", drifts, flush=True)

    if "cfg5" in which:
        cond, text, y0, N, kw = inputs_cfg5()
        t0 = time.time()
        with torch.no_grad():
            out, traj = O.sample(cond, text, N, W, ocfg, y0=y0, **kw)
            out16, _ = O.sample(cond, text, N, W, ocfg, y0=y0, prec=emu, **kw)
            # one forward at an interior time (text positions beyond 4095 reuse the last row, rope.py:83)
            prep = O.sample_prologue(cond, text, N, W, max_duration=8192)
            tt = torch.tensor(0.25)
            fwd = O.dit_forward(y0, prep.step_cond, prep.text, tt, False, False, None, W, ocfg)
            fwd16 = O.dit_forward(y0, prep.step_cond, prep.text, tt, False, False, None, W, ocfg, emu)
        drift = _rel(out16[:, NREF60S:], out[:, NREF60S:])
        # every 6th frame of the sample and of the forward keeps the file under 1 MB
        np.savez_compressed(os.path.join(HERE, "full_cfg5_long.npz"), out_sub6=out[0, ::6].numpy(), drift=np.float64(drift),
                            fwd_sub6=fwd[0, ::6].numpy(), fwd_drift=np.float64(_rel(fwd16, fwd)), weight_seed=1234,
                            input_seed=50505, input_checksum=input_checksum(cond, text, y0))
        print(f"cfg5: {time.time() - t0:.0f}s drift={drift:.3e} fwd drift={_rel(fwd16, fwd):.3e}", flush=True)
    for f in sorted(os.listdir(HERE)):
        if f.startswith("full_"):
            print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == "__main__":
    main()
