#!/usr/bin/env python
"""bench.py — mel-frames/sec of the F5TTS.sample() hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one F5TTS.sample() ODE solve of one batch of synthetic utterances per GPU
(default workload = BASELINE.json configs[1]: F5-TTS base 22-layer/1024-dim/16-head DiT, 10 s
utterance = 937 mel frames (328 ref + 609 gen), 152 text tokens, Euler, steps=32 grid points
(31 intervals, 62 DiT evaluations with CFG=2), batch 1 per GPU).  Weights are seeded random
(no checkpoints are reachable), inputs synthetic.

  value      : whole-job mel-frames/s, inputs resident in HBM (CUDA-graph replay of the loop)
  e2e        : same metric through the public API a user calls — F5TTS.sample(raw wave on the
               HOST, text) -> waveform on the HOST: H2D of the reference audio + noise, log-mel
               front-end, ODE loop, Vocos vocoder, D2H of the waveform, all inside the timed region
  roofline   : tcgen05 GEMM family (the dominant kernels): algorithmic FLOPs / summed in-situ duration
               of its launches INSIDE the replayed CUDA graph (per-launch %globaltimer stamps: first
               CTA past the dependency wait -> last CTA exit), so family time <= ms_per_step
  configs    : BASELINE configs 3 (64 x 10 s, midpoint; = config 4 at --gpus 8) and 5 (60 s long-form)
               measured the same way, each with its own roofline
  cpu_baseline: the CPU oracle (torch-CPU fp32 restatement of the reference — MLX itself is not
               installable here) timed on this box's host cores on a bounded sample of the SAME
               workload
  --impl reference : times only that CPU restatement (rank 0), same metric/config.
  --steps K  : timed steps of the headline, of e2e and of the FP8 mode (configs 3 and 5 time 2 and 3 steps)
  --dump-outputs DIR : what the last timed step of each of them returned, as DIR/<name>.npy (see dump_outputs);
               inputs and weights are seeded, so two builds run with the same arguments compare output for output
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR, HOP = 24000, 256
TOTAL_SAMPLES, REF_SAMPLES, N_TEXT = 240000, 84000, 152      # SURVEY §8d synthetic "10 s" utterance


def synth_audio(length: int, seed: int) -> torch.Tensor:
    rng = np.random.default_rng(seed)
    t = np.arange(length) / SR
    f0 = 110 + 110 * rng.random()
    x = sum(np.sin(2 * np.pi * f0 * (h + 1) * t + rng.random() * 6.28) / (h + 1) for h in range(8))
    x = x * (0.6 + 0.4 * np.sin(2 * np.pi * 1.3 * t)) + 0.01 * rng.standard_normal(length)
    return torch.from_numpy((x * 0.1 / np.sqrt(np.mean(x ** 2))).astype(np.float32))


def synth_inputs(batch: int, frames: int, ref_frames: int, seed: int):
    g = torch.Generator().manual_seed(seed)
    cond = (torch.randn(batch, ref_frames, 100, generator=g) * 2.24 - 1.27).clamp(-11.51, 5.0)
    text = torch.randint(0, 2545, (batch, N_TEXT), generator=g, dtype=torch.int32)
    y0 = torch.randn(batch, 100, frames, generator=g).permute(0, 2, 1).contiguous()
    return cond, text, y0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,clocks.mem,clocks.max.mem")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, mem, pw = [], [], set(), [], []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            try:
                pw.append(float(r[3])); mem.append(float(r[8]))
            except Exception:
                pass
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "mem_mhz": statistics.median(mem) if mem else None,
                "power_w": statistics.median(pw) if pw else None}


def ncu_traffic() -> dict:
    """DRAM bytes per launch of the dominant (GEMM) kernels from the committed `ncu --set full` captures of this
    workload (profiles/*_ncu_full.json, see tools/profile.sh): cold (ncu flushes the caches before every replay) and,
    when captured, warm (--cache-control none: activations L2-resident as inside a step); None if absent."""
    import glob, re
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_full.json")))
    if not files:
        return {"traffic": None}

    def dram(rec):
        tot = 0.0
        for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            m = re.match(r"([0-9.,]+)\s*(\w*)", rec.get(k, "0 byte"))
            tot += float(m.group(1).replace(",", "")) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(m.group(2), 1)
        return tot
    try:
        d = json.load(open(files[-1]))
        cold = [dram(r) for k, v in d.items() if k.startswith("gemm") and "warm" not in k for r in v]
        warm = [dram(r) for k, v in d.items() if k.startswith("gemm") and "warm" in k for r in v]
        if not cold:
            return {"traffic": None}
        out = {"traffic": sum(cold) / len(cold),
               "traffic_note": f"mean DRAM read+write bytes per launch over the {len(cold)} block-GEMM launches captured in "
                               f"{os.path.basename(files[-1])} (cold cache under ncu)"}
        if warm:
            out["traffic_warm"] = sum(warm) / len(warm)
        return out
    except Exception as e:  # pragma: no cover
        return {"traffic": None, "traffic_note": f"unreadable profile: {e}"}


def peaks() -> dict:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "hbm_gbs": d.get("hbm_gbs"),
                "source": "MEASURED_PEAKS.json (bf16_tflops_sustained: kernels timed inside a long step)"}
    return {"bf16_tflops": 1400.0, "hbm_gbs": 6650.0, "source": "fallback of B200_PROFILING.md (sustained 1.4 PF)"}


# ---------------------------------------------------------------------------------------------
# CPU oracle leg (cpu_baseline / --impl reference)
# ---------------------------------------------------------------------------------------------
def oracle_step(args, W, ocfg, intervals: int, seed: int):
    """Bounded sample of the workload: `intervals` solver intervals of ONE utterance of the same
    shape, run exactly like the reference (two unbatched CFG passes, text embedding per forward).
    Returns (seconds, frames/s extrapolated to the full grid)."""
    from oracle import f5_oracle as O
    frames, ref_frames = args.frames, args.ref_frames
    cond, text, y0 = synth_inputs(1, frames, ref_frames, seed)
    full_t = O.time_grid(args.ode_steps, -1.0)
    prep = O.sample_prologue(cond, text, frames, W)
    solver = {"euler": O.odeint_euler, "midpoint": O.odeint_midpoint, "rk4": O.odeint_rk4}[args.method]

    def fn(t, x):
        pred = O.dit_forward(x, prep.step_cond, prep.text, t, False, False, prep.mask, W, ocfg)
        null = O.dit_forward(x, prep.step_cond, prep.text, t, True, True, prep.mask, W, ocfg)
        return pred + (pred - null) * args.cfg

    t0 = time.perf_counter()
    with torch.no_grad():
        solver(fn, y0, full_t[: intervals + 1])
    dt = time.perf_counter() - t0
    full = dt * (args.ode_steps - 1) / intervals
    return dt, frames / full


def pick_cpu_threads() -> int:
    """"All the host threads it can use": a many-core host is SLOWER with one thread per core on
    these matmul sizes (first run on the 128-core GPU box: 0.43 frames/s with 128 threads), so time
    the dominant GEMM shape at a few thread counts and keep the fastest."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 48, 64, 96, ncpu) if c <= ncpu})
    a, b = torch.randn(1874, 1024), torch.randn(2048, 1024)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        torch.mm(a, b.T)
        t0 = time.perf_counter()
        for _ in range(5):
            torch.mm(a, b.T)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def oracle_setup(args):
    from oracle import f5_oracle as O
    from f5_tts_mlx_b200.weights import BASE_CONFIG, random_dit_weights
    pick_cpu_threads()
    cfg = BASE_CONFIG
    W = random_dit_weights(cfg, seed=1234)
    ocfg = O.DiTConfig(dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, ff_mult=cfg.ff_mult,
                       text_num_embeds=cfg.text_num_embeds, text_dim=cfg.text_dim, conv_layers=cfg.conv_layers)
    return W, ocfg


def run_reference(args, rank: int, world: int):
    """The reference's own CPU path for the same metric/config (rank 0 only; other ranks exit 0 without work).
    MLX is not installable here, so this is the oracle — the torch-CPU restatement pinned to the unmodified reference
    sources through tests/mlx_shim.  One step = a BOUNDED sample: `intervals` of the solver's intervals of ONE
    utterance of the workload, extrapolated to the full grid.  Utterances are independent (cfm.py:340-365) and the
    reference runs them in one process, so its frames/s for the global batch is the per-utterance figure — which is
    why `config` (global_batch = batch x n_gpus) is the CUDA arm's and the value does not grow with --gpus."""
    if rank != 0:
        return
    W, ocfg = oracle_setup(args)
    intervals = 2
    steps_run = min(args.steps, 10)          # each step is ~8-20 s of CPU: keep the whole run within minutes
    for _ in range(args.warmup):
        oracle_step(args, W, ocfg, 1, 0)
    times, fps = [], []
    for i in range(steps_run):
        dt, f = oracle_step(args, W, ocfg, intervals, i)
        times.append(dt); fps.append(f)
    val = args.frames * len(fps) / sum(args.frames / f for f in fps)
    cores = torch.get_num_threads()
    sample = (f"{intervals} of {args.ode_steps - 1} {args.method} intervals ({2 * intervals} DiT evaluations with CFG) of ONE "
              f"{args.frames}-frame utterance per step, extrapolated x{(args.ode_steps - 1) / intervals:.1f} to the full grid; "
              f"{steps_run} such steps run (requested {args.steps}, capped at 10); per-utterance rate = rate for the "
              f"global batch of {args.batch * world} (independent utterances, one CPU process)")
    wl = Workload("main", args.batch, args.frames, args.ref_frames, args.method, args.ode_steps, args.cfg)
    line = {"impl": "reference", "metric": "mel-frames/sec", "value": val, "unit": "mel-frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "steps_run": steps_run, "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(times),
            "ms_per_step_is": "one bounded sample (see cpu_baseline.sample), not a full utterance",
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": wl.describe(world),
            "cpu_baseline": {"value": val, "unit": "mel-frames/s", "cores": cores, "kind": "port",
                             "sample": sample + f"; threads chosen by a GEMM calibration out of {os.cpu_count()} logical CPUs",
                             "note": "torch-CPU fp32 restatement of the reference (oracle/f5_oracle.py), pinned to the "
                                     "reference's own code via tests/mlx_shim; MLX is not installable in this image"},
            "e2e": {"value": val, "unit": "mel-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# CUDA arm
# ---------------------------------------------------------------------------------------------
class Workload:
    """One (batch, frames, solver) point: synthetic inputs resident in HBM, the captured CUDA graph of
    precompute + ODE loop with in-graph timing slots, and its measurement."""

    def __init__(self, name, batch, frames, ref_frames, method, ode_steps, cfg, n_text=N_TEXT, extra=None):
        self.name, self.batch, self.frames, self.ref_frames = name, batch, frames, ref_frames
        self.method, self.ode_steps, self.cfg, self.n_text = method, ode_steps, cfg, n_text
        self.extra = extra or {}

    def describe(self, world: int) -> dict:
        return {"workload": f"F5-TTS base DiT 22L/1024d/16h, {self.batch} x {self.frames * HOP / SR:.0f} s utterance per GPU "
                            f"({self.frames} mel frames = {self.ref_frames} ref + {self.frames - self.ref_frames} gen, "
                            f"{self.n_text} text tokens), {self.method} steps={self.ode_steps} grid points "
                            f"({self.ode_steps - 1} intervals), CFG={self.cfg}, sway=-1",
                "global_batch": self.batch * world, "frames": self.frames, "parallelism": f"dp{world}",
                "l2": "no flush: the 0.67 GB of bf16 weights streamed every DiT evaluation exceed the 126 MB L2"}


def measure(f5, lib, wl: Workload, rank: int, world: int, dev, steps: int, warmup: int, clocks=None) -> dict:
    """Timed region = `steps` graph replays (inputs resident); then ONE more replay with the in-graph timing slots
    reset, from which the per-family device times come (same graph, same stream, inside the step)."""
    import ctypes as C
    import torch.distributed as dist
    B, N, NR = wl.batch, wl.frames, wl.ref_frames
    g = torch.Generator().manual_seed(100 + rank + 17 * B + N)
    cond = (torch.randn(B, NR, 100, generator=g) * 2.24 - 1.27).clamp(-11.51, 5.0)
    text = torch.randint(0, 2545, (B, wl.n_text), generator=g, dtype=torch.int32)
    y0 = torch.randn(B, 100, N, generator=g).permute(0, 2, 1).contiguous()
    cond_d, y0_d = cond.to(dev), y0.to(dev)
    kw = dict(steps=wl.ode_steps, method=wl.method, cfg_strength=wl.cfg, sway_sampling_coef=-1.0, return_trajectory=False)
    if N > 4096:
        kw["max_duration"] = N        # long-form (config 5): the reference's default clip is 4096 frames (cfm.py:277)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # eager pass (sets kernel attributes, validates), launch count, then capture WITH timing slots installed
    f5.use_cuda_graph = False
    c0 = lib.f5_launch_count()
    out, _ = f5.sample(cond_d, text, N, y0=y0_d, **kw)
    torch.cuda.synchronize()
    launches_per_step = int(lib.f5_launch_count() - c0)
    assert torch.isfinite(out).all().item(), "non-finite output"
    plan = f5.last_plan
    f5.use_cuda_graph = True
    cap = launches_per_step + 64
    slots = torch.zeros(cap, 2, dtype=torch.int64, device=dev)
    lib.f5_prof_graph_begin(C.c_void_p(slots.data_ptr()), cap)
    plan.capture(f5)
    lib.f5_prof_graph_begin(None, 0)
    kinds = (C.c_int32 * cap)(); flops = (C.c_double * cap)(); nbytes = (C.c_double * cap)()
    n_slots = lib.f5_prof_graph_meta(kinds, flops, nbytes, cap)

    def step():
        plan.y.copy_(y0_d)
        plan.graph.replay()

    for _ in range(max(warmup, 3) if steps > 3 else max(warmup, 1)):
        step()
    barrier()
    if clocks is not None:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    # what sample() returns for the last timed step: the final ODE state and the mel with the reference frames put back
    state = plan.y[:, :N].clone()
    mel = state.clone()
    mel[:, :NR] = cond_d
    clk = clocks.stop() if clocks is not None else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = t.item() / steps

    # in-graph per-family device time: one replay with the slots reset
    slots[:, 0] = -1          # UINT64_MAX
    slots[:, 1] = 0
    step()
    torch.cuda.synchronize()
    sl = slots[:n_slots].cpu().numpy()
    fam = {k: {"ms": 0.0, "flops": 0.0, "launches": 0} for k in ("gemm", "attention")}
    for i in range(n_slots):
        k = kinds[i]
        if k > 1 or sl[i, 0] == -1 or sl[i, 1] == 0:
            continue
        f = fam["gemm" if k == 0 else "attention"]
        f["ms"] += (int(sl[i, 1]) - int(sl[i, 0])) * 1e-6
        f["flops"] += flops[i]; f["launches"] += 1

    pk = peaks()
    from oracle import f5_oracle as O
    ocfg = O.DiTConfig()
    n_fwd = O.dit_forwards_per_sample(wl.ode_steps, wl.method, wl.cfg)
    alg = n_fwd * O.dit_forward_flops(N, ocfg) * B
    gm, at = fam["gemm"], fam["attention"]
    ach = gm["flops"] / (gm["ms"] * 1e-3) / 1e12 if gm["ms"] > 0 else 0.0
    roof = {"bound": "tensor", "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"],
            **ncu_traffic(),
            "kernel": "gemm_bf16_tn_kernel + gemm2_bf16_tn_kernel (tcgen05; every GEMM launch of one step)",
            "how": "per-launch in-situ duration inside the replayed CUDA graph: min over CTAs of %globaltimer after the "
                   "dependency wait -> max over CTAs at exit, summed over the family; algorithmic 2MNK flops",
            "of": pk["source"], "gemm_ms_per_step": gm["ms"], "gemm_launches_per_step": gm["launches"],
            "gemm_share_of_step": gm["ms"] / ms_step if ms_step else None,
            "attention": {"achieved": at["flops"] / (at["ms"] * 1e-3) / 1e12 if at["ms"] > 0 else 0.0, "ms_per_step": at["ms"],
                          "share_of_step": at["ms"] / ms_step if ms_step else None, "launches_per_step": at["launches"]},
            "other_ms_per_step": ms_step - gm["ms"] - at["ms"],
            "whole_step": {"algorithmic_tflop": alg / 1e12, "achieved_tflops_per_gpu": alg / (ms_step * 1e-3) / 1e12,
                           "frac": alg / (ms_step * 1e-3) / 1e12 / pk["bf16_tflops"]}}
    res = {"ms_per_step": ms_step, "value": world * B * N / (ms_step / 1e3), "unit": "mel-frames/s", "steps": steps,
           "launches_per_step": launches_per_step, "roofline": roof, "config": wl.describe(world),
           "rtf": (ms_step / 1e3) / (B * (N - NR) * HOP / SR), "generated_frames_per_s": world * B * (N - NR) / (ms_step / 1e3)}
    if clk is not None:
        res["clocks"] = clk
    res["_inputs"] = (cond, text, y0, kw)
    res["_outputs"] = {"mel": mel, "trajectory": state[None]}
    return res


def run_cuda(args, rank: int, world: int, local_rank: int):
    import torch.distributed as dist
    from f5_tts_mlx_b200 import BASE_CONFIG, DiT, F5TTS, _lib
    from f5_tts_mlx_b200.vocos import Vocos
    from f5_tts_mlx_b200.weights import VocosConfig, random_dit_weights, random_vocos_weights

    if not torch.cuda.is_available():
        # the product path has no CPU fallback: say so instead of measuring something else
        sys.stderr.write("bench.py: no CUDA device visible; this arm runs libf5b200.so on a B200 only "
                         "(the CPU baseline is `--impl reference`)\n")
        raise SystemExit(3)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _lib.load()
    cfg = BASE_CONFIG
    model = DiT(dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, ff_mult=cfg.ff_mult, mel_dim=cfg.mel_dim,
                text_num_embeds=cfg.text_num_embeds, text_dim=cfg.text_dim, conv_layers=cfg.conv_layers, device=dev,
                fused_adaln=not args.no_fused_adaln, fp8=args.fp8)
    # rank 0 builds + packs the weights; ONE broadcast of the packed buffer (the only collective)
    if rank == 0:
        model.load_weights(random_dit_weights(cfg, seed=1234))
    else:
        model.allocate_weights()
    if world > 1:
        model.packed.broadcast(src=0)
    vocos = Vocos(VocosConfig(), dev).load_weights(random_vocos_weights())
    f5 = F5TTS(model)
    f5_e2e = F5TTS(model, vocoder=vocos.decode)

    B, N, NR = args.batch, args.frames, args.ref_frames
    main_wl = Workload("main", B, N, NR, args.method, args.ode_steps, args.cfg)

    if args.profile_run:
        # under ncu: one eager pass of the same step, then the audio front-end and the vocoder (nothing is timed)
        g = torch.Generator().manual_seed(100)
        cond = (torch.randn(B, NR, 100, generator=g) * 2.24 - 1.27).clamp(-11.51, 5.0).to(dev)
        text = torch.randint(0, 2545, (B, N_TEXT), generator=g, dtype=torch.int32)
        kw = dict(steps=args.ode_steps, method=args.method, cfg_strength=args.cfg, sway_sampling_coef=-1.0, return_trajectory=False)
        if N > 4096:
            kw["max_duration"] = N
        f5.use_cuda_graph = False
        f5_e2e.use_cuda_graph = False
        # first the audio front-end + a 2-grid-point sample + the vocoder (so the mel / ISTFT / Vocos kernels are
        # among the first launches of the list), then the full step
        audio = synth_audio(REF_SAMPLES, seed=7).to(dev)
        f5_e2e.sample(audio[None], text[:1], N, seed=0, **{**kw, "steps": 2})
        f5.sample(cond, text, N, seed=0, **kw)
        torch.cuda.synchronize()
        return

    clocks = ClockSampler(local_rank)
    m = measure(f5, lib, main_wl, rank, world, dev, args.steps, args.warmup, clocks)
    cond, text, y0, kw = m.pop("_inputs")
    outputs = m.pop("_outputs")

    # ---- end to end through the public API with HOST buffers (same batch as the headline) ----
    e2e_steps = args.steps
    y0_h = y0.contiguous().pin_memory()
    if B == 1:
        audio_h = synth_audio(REF_SAMPLES if NR == REF_SAMPLES // HOP else NR * HOP, seed=7 + rank).pin_memory()
        cond_h = audio_h[None]          # raw wave (1, samples): the mel front-end runs inside sample() (cfm.py:283-286)
        path = "F5TTS.sample(host raw wave, text) -> mel kernel -> ODE loop -> Vocos -> host waveform"
    else:
        cond_h = cond.contiguous().pin_memory()     # raw-wave conditioning is batch-1 only in the reference (cfm.py:284)
        path = "F5TTS.sample(host mel batch, text) -> ODE loop -> Vocos (batched) -> host waveforms"

    def e2e_once():
        c = cond_h.to(dev, non_blocking=True)
        wave, _ = f5_e2e.sample(c, text, N, y0=y0_h.to(dev, non_blocking=True), **kw)
        return wave.to("cpu", non_blocking=False)

    for _ in range(3):
        w = e2e_once()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        w = e2e_once()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    outputs["e2e_wave"] = w
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = world * B * N * e2e_steps / te.item()
    h2d = cond_h.numel() * 4 + y0_h.numel() * 4 + text.numel() * 4
    d2h = w.numel() * 4

    # ---- the other BASELINE configurations as sub-results of the same line (each with its own roofline) ----
    subs = {}
    if not args.no_configs and B == 1 and N == TOTAL_SAMPLES // HOP:
        for wl, st in ((Workload("cfg3_b64_midpoint", 64, N, NR, "midpoint", 32, 2.0), 2),
                       (Workload("cfg5_long60s", 1, 5625, 499, "euler", 32, 2.0, n_text=N_TEXT * 6), 3)):
            f5._plans.clear(); model._sessions.clear(); torch.cuda.empty_cache()
            r = measure(f5, lib, wl, rank, world, dev, st, 1)
            r.pop("_inputs")
            outputs[wl.name + "_mel"] = r.pop("_outputs")["mel"]
            subs[wl.name] = r
        # config 4 of BASELINE.json (512 utterances over 8 GPUs = 64 per GPU, weights broadcast once, no per-step
        # collective) is cfg3_b64_midpoint at --gpus 8: its `value` is the whole-job aggregate over all ranks
        subs["cfg3_b64_midpoint"]["note"] = (f"global batch {64 * world} utterances over {world} GPU(s); at --gpus 8 this is "
                                             "BASELINE config 4 (512 utterances sharded 64 per GPU)")
        f5._plans.clear(); model._sessions.clear(); torch.cuda.empty_cache()
        if not args.fp8:
            # the headline workload in FP8 mode (e4m3 operands on the four GEMMs of every block): the lossy analogue of
            # the reference's quantised `--q` checkpoints, reported beside the bf16 headline, never instead of it
            m8 = DiT(dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, ff_mult=cfg.ff_mult, mel_dim=cfg.mel_dim,
                     text_num_embeds=cfg.text_num_embeds, text_dim=cfg.text_dim, conv_layers=cfg.conv_layers, device=dev, fp8=True)
            if rank == 0:
                m8.load_weights(random_dit_weights(cfg, seed=1234))
            else:
                m8.allocate_weights()
            if world > 1:
                m8.packed.broadcast(src=0)
            r = measure(F5TTS(m8), lib, Workload("b1_fp8", B, N, NR, args.method, args.ode_steps, args.cfg), rank, world, dev,
                        args.steps, 3)
            r.pop("_inputs")
            outputs["b1_fp8_mel"] = r.pop("_outputs")["mel"]
            r["dtype"] = "fp8 (e4m3 operands of QKV / out / FF1 / FF2, fp32 accumulate) + bf16 elsewhere"
            r["note"] = "lossy mode: oracle-emulated drift 2.9e-2 per forward vs 3.9e-3 for bf16 (DESIGN.md section 8)"
            subs["b1_fp8"] = r
            del m8
            torch.cuda.empty_cache()

    if rank != 0:
        return
    # CPU baseline beside it (bounded sample)
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        W, ocfg2 = oracle_setup(args)
        oracle_step(args, W, ocfg2, 1, 0)
        dt, fps = oracle_step(args, W, ocfg2, 2, 1)
        cpu = {"value": fps, "unit": "mel-frames/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"2 of {args.ode_steps - 1} {args.method} intervals (4 DiT evaluations) of one {N}-frame utterance "
                         f"({dt:.1f} s of CPU), extrapolated to the full grid; threads chosen by a GEMM calibration "
                         f"out of {os.cpu_count()} logical CPUs",
               "note": "torch-CPU fp32 restatement of the reference, pinned to the reference's own code through "
                       "tests/mlx_shim (MLX itself is not installable in this image)"}
    line = {"metric": "mel-frames/sec", "value": m["value"], "unit": "mel-frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": m["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp8(e4m3 QKV/FF1)+bf16" if args.fp8 else "bf16", "data": "synthetic",
            "config": m["config"], "clocks": m.get("clocks"),
            "e2e": {"value": e2e_val, "unit": "mel-frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "path": path, "ms_per_step": 1e3 * te.item() / e2e_steps, "batch": B},
            "gpu_launches": m["launches_per_step"] * args.steps, "launches_per_step": m["launches_per_step"],
            "roofline": m["roofline"], "cpu_baseline": cpu, "rtf": m["rtf"],
            "generated_frames_per_s": m["generated_frames_per_s"], "fused_adaln": not args.no_fused_adaln,
            "configs": subs}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes rank 0's outputs of the last timed step as <out_dir>/<name>.npy in float32, DUMP_BYTES at most in all:
    the smaller arrays are written whole, and one whose share of what is left is too small is replaced by a fixed,
    seeded sample of its elements (flattened, in index order), so two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    left = DUMP_BYTES
    for i, (name, t) in enumerate(items):
        a = t.detach().float().cpu().numpy()
        keep = (left // (len(items) - i) - 128) // a.itemsize           # 128: the .npy header
        if a.size > keep:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, a)
        left -= os.path.getsize(path)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--batch", type=int, default=1, help="utterances per GPU per step")
    ap.add_argument("--frames", type=int, default=TOTAL_SAMPLES // HOP)
    ap.add_argument("--ref-frames", type=int, default=REF_SAMPLES // HOP)
    ap.add_argument("--ode-steps", type=int, default=32)
    ap.add_argument("--method", default="euler", choices=["euler", "midpoint", "rk4"])
    ap.add_argument("--cfg", type=float, default=2.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the config-3 / config-5 sub-results")
    ap.add_argument("--no-fused-adaln", action="store_true", help="A/B: separate LayerNorm+modulate launches (r01 path)")
    ap.add_argument("--fp8", action="store_true", help="FP8 mode (e4m3 QKV / FF1 GEMMs): the lossy analogue of the reference's --q; "
                                                        "NOT the headline (dtype is reported as fp8+bf16)")
    ap.add_argument("--profile-run", action="store_true", help="one eager step and exit (for ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (mel, trajectory, e2e_wave, <config>_mel) "
                         "as DIR/<name>.npy, float32, 64 MB at most")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.profile_run):
        ap.error("--dump-outputs applies to the timed CUDA arm")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_cuda(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
