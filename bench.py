#!/usr/bin/env python
"""bench.py — env-steps/sec of the batched xLSTM recurrent inference step (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--model 48M] [--envs 64]
                    [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] — "xLSTM 48M recurrent step, 64 synthetic Meta-World envs
on 1xB200"; for N > 1 every rank runs the same 64 envs-per-GPU shard (weak scaling; env i -> rank i % N as
`custom_eval_callback.py:385`), weights replicated, state cache per GPU, ONE all_gather of the int32 action tokens
per step. A "step" is one env step of all envs: embed + 3 tokens x 12 blocks + head + argmax/inv_tokenize.

  value        env-steps/s, inputs (the whole synthetic stream) resident in HBM before the timed region
  e2e          same metric through the C-ABI host call xl_policy_step_host: pinned host buffers, H2D of the step's
               states/rtg and D2H of tokens+actions inside the timed region, one stream sync per step
  roofline     the mLSTM state-step kernel: algorithmic C/n/m bytes per launch / average launch duration, timed
               with CUDA events around each of its launches in a profiled replay of the same steps
  whole_step   the un-gameable figure: algorithmic bytes of the WHOLE env step (state of every block once + weights)
               / the graph-timed step, against the same measured peak
  cpu_baseline the oracle (restated xlstm native PyTorch path, fp32) on the box's host cores, bounded sample
  gpu_eager_baseline  the same oracle op sequence run eagerly on the GPU (fp32, ~10^3 launches per env step): the
               like-for-like "reference on this GPU" comparator (what `inf_dummy_batch_size` measures in the
               reference, online_decision_transformer_model.py:748-758)
  context_prefill  BASELINE.json configs[3] on the side (N = 1): 49 998-token chunkwise prefill of one 206M env, tokens/s
               and the bf16 MMA rate of the whole prefill against the sustained cuBLAS rate (tensor-pipe utilisation)

--dump-outputs DIR: after the timed steps, writes what the last of them returned to its caller as DIR/<name>.npy
(float32 / float64; the inputs are seeded, so two builds run with the same arguments can be compared file for file):
action_tokens and action_preds of every env of this rank, and a fixed seeded sample (48 MiB at most) of the recurrent
state every block carries into the next step, state_block<i>_<C|n|m|conv|slstm>.npy (C in the reference's
[B, NH, DH, DH] layout, flattened).

--impl reference: times the reference's CPU implementation of the path (the oracle port; the xlstm package is
absent, see oracle/xlstm_oracle.py header) on the host cores for the same config/metric. Both CPU legs use ONE
sample definition (cpu_sample): the first min(envs, 8) envs of the workload, all host threads.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "env-steps/sec batched xLSTM recurrent inference"
UNIT = "env-steps/s"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return json.load(fh), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def mark(self):
        """samples read from here on belong to the measured window"""
        self.lines = []

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def workload_config(args, world):
    """The workload both arms are measured on (BASELINE.json configs[1] by default)."""
    B = args.envs
    return {"workload": f"xLSTM {args.model} recurrent step, {B} synthetic {args.domains} envs per GPU"
                        + (" (BASELINE.json configs[1])" if (args.model, B) == ("48M", 64) else ""),
            "model": args.model, "envs_per_gpu": B, "global_envs": B * world, "tokens_per_step": 3,
            "domains": args.domains, "head": "discrete" if args.discrete else "continuous-tokenized"}


CPU_SAMPLE_ENVS = 8


def cpu_sample(envs: int) -> int:
    """The ONE bounded sample both CPU legs (cpu_baseline and --impl reference) time: the first min(envs, 8) envs of
    the workload (batch rows are independent; per-env cost on the CPU is, if anything, lower at 8 envs than at 64,
    whose 1.75 GB of state no longer fits the host caches — so the sample flatters the CPU, not the GPU)."""
    return min(envs, CPU_SAMPLE_ENVS)


def time_oracle(cfg, sd, B, n_steps, warmup, threads, budget_s=None, domains="metaworld", discrete=False,
                device="cpu"):
    """Oracle env steps on the host cores (or, device="cuda", the same eager op sequence on the GPU).
    Returns (env_steps_per_s, ms list, steps actually timed)."""
    from lram_b200.synth import make_stream
    from oracle.xlstm_oracle import OraclePolicy
    torch.set_num_threads(threads)
    pol = OraclePolicy(cfg, sd, device=device)
    states, rtg, _ = make_stream(cfg, range(B), min(n_steps + warmup, 64), domains=domains)
    d_states, d_rtg = torch.from_numpy(states).to(device), torch.from_numpy(rtg).to(device)
    pkv = None
    ms = []
    t_begin = time.perf_counter()
    for t in range(n_steps + warmup):
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        o = pol.step(d_states[t % len(states)], d_rtg[t % len(states)], past_key_values=pkv, discrete=discrete)
        if device != "cpu":
            o["action_tokens"].cpu()                      # the rollout reads the action on the host (evaluation.py:141)
        pkv = o["past_key_values"]
        dt = time.perf_counter() - t0
        if t >= warmup:
            ms.append(dt * 1e3)
            if budget_s is not None and time.perf_counter() - t_begin > budget_s and len(ms) >= 2:
                break
    total = sum(ms) / 1e3
    return B * len(ms) / total, ms, len(ms)


def run_reference(args):
    """`--impl reference`: the reference's own CPU execution mode for this path (xlstm native PyTorch ops, fp32),
    i.e. the oracle port, on all host cores. Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from lram_b200.config import preset
    from lram_b200.synth import make_state_dict
    if args.scaling == "strong":                      # --envs is the job's env count: per-GPU share, as the b200 arm
        args.envs = args.envs // max(args.gpus, 1)
    cfg = preset(args.model)
    sd = make_state_dict(cfg, seed=0)
    cores = os.cpu_count() or 1
    # bounded sample (the same definition as the b200 arm's cpu_baseline): cpu_sample(envs) envs, every step one env
    # step of those envs; exactly K timed steps
    b_ref = cpu_sample(args.envs)
    kw = dict(domains=args.domains, discrete=args.discrete)
    value, ms, timed = time_oracle(cfg, sd, b_ref, args.steps, args.warmup, cores, **kw)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": timed, "warmup": args.warmup, "ms_per_step": statistics.mean(ms), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # global_envs is what THIS arm ran (the bounded sample on rank 0), not the N-GPU job's env count
        "config": dict(workload_config(args, max(args.gpus, 1)), global_envs=b_ref, backend="oracle port of the "
                       "xlstm native PyTorch ops, CPU fp32, rank 0 only", sampled_envs=b_ref,
                       job_envs=args.envs * max(args.gpus, 1)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{b_ref} of {args.envs} envs x {timed} env steps, oracle port of the xlstm "
                                   f"native PyTorch backend (xlstm package absent), fp32, {cores} threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)


_JSON_FD = None


def prefill_leg(peaks, model="206M", tokens=49998, reps=2):
    """BASELINE.json configs[3]: chunkwise context prefill of one env (tcgen05 cell + tcgen05 projections), timed with
    CUDA events over whole xl_policy_prefill calls (inputs resident in HBM). `tensor` relates the bf16 MMA work the
    prefill issues (hi/lo passes included) to the sustained cuBLAS bf16 rate of MEASURED_PEAKS.json."""
    from lram_b200.config import preset
    from lram_b200.engine import XLSTMEngine
    from lram_b200.synth import make_state_dict, make_stream
    cfg = preset(model)
    sd = make_state_dict(cfg, seed=0)
    eng = XLSTMEngine(cfg, sd, max_batch=1)
    Tn = tokens // 3
    st_np, rtg_np, _ = make_stream(cfg, range(1), 256, domains="mixed")
    rep = (Tn + 255) // 256
    states = torch.from_numpy(np.ascontiguousarray(np.tile(st_np, (rep, 1, 1))[:Tn].transpose(1, 0, 2))).cuda()
    rtg = torch.from_numpy(np.ascontiguousarray(np.tile(rtg_np, (rep, 1))[:Tn].T)).cuda()
    cache = eng.new_state(1)
    times = []
    for r in range(reps + 1):
        eng.reset(cache)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.policy_prefill(cache, states, rtg)
        e1.record()
        torch.cuda.synchronize()
        if r > 0:                                   # the first call allocates the prefill workspaces
            times.append(e0.elapsed_time(e1))
    eng.close()
    ms = statistics.median(times)
    S, d, inner, NH, DH, Lb = Tn * 3, cfg.d, cfg.inner, cfg.num_heads, cfg.head_dim, cfg.num_blocks
    proj = 2 * (2.0 * S * d * 2 * inner + 2.0 * S * inner * d)                       # A = hi + lo: two MMA passes
    chunks = (S + 127) // 128
    cell = 3 * chunks * NH * (2.0 * DH * DH * 128 + 2.0 * 128 * 128 * DH + 2.0 * 128 * DH * (DH + 128))   # hi/lo x hi/lo
    mma = Lb * (proj + cell)
    peak = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops")
    return {"workload": f"xLSTM {model}, 1 env, {S}-token context (chunkwise prefill, then O(1) recurrent rollout)",
            "tokens_per_s": S / (ms / 1e3), "ms": ms, "reps": reps,
            "tensor": {"bound": "tensor", "achieved": mma / (ms / 1e3) / 1e12, "peak": peak, "unit": "TFLOP/s",
                       "frac": mma / (ms / 1e3) / 1e12 / peak if peak else None,
                       "note": "bf16 MMA flops issued by the projections (2 passes) and the chunkwise cell (3 passes) "
                               "over the WHOLE prefill time, non-GEMM kernels included; peak = sustained cuBLAS bf16"}}


DUMP_STATE_BYTES = 48 * 2 ** 20


def snapshot_outputs(cfg, out, cache) -> dict:
    """Device copies of what a policy step returned to its caller (see --dump-outputs), keyed by file name. They stay
    on the device so that the copy to the host can wait until the clock-sampling window has closed."""
    from lram_b200 import _lib as L
    arrays = {"action_tokens": out["action_tokens"].double(),                     # int32 values, exact in float64
              "action_preds": out["action_preds"].float().clone()}
    parts = []
    for i in range(cfg.num_blocks):
        if cfg.is_slstm(i):
            parts += [(i, "slstm", L.XL_STATE_SLSTM), (i, "conv", L.XL_STATE_CONV)]
        else:
            parts += [(i, "C", None), (i, "n", L.XL_STATE_N), (i, "m", L.XL_STATE_M), (i, "conv", L.XL_STATE_CONV)]
    cap = DUMP_STATE_BYTES // 4 // len(parts)
    g = torch.Generator().manual_seed(0)
    for i, name, part in parts:
        t = (cache.c_logical(i) if part is None else cache.view(i, part)).reshape(-1)
        if t.numel() > cap:
            idx = torch.randint(t.numel(), (cap,), generator=g).sort().values
            t = t[idx.to(t.device)]
        arrays[f"state_block{i:02d}_{name}"] = t.float().clone()
    return arrays


def _quiet_stdout():
    """The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version banner from C), so
    fd 1 is pointed at stderr for the whole run and the JSON line goes to a duplicate of the original stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="48M")
    ap.add_argument("--envs", type=int, default=64, help="envs per GPU")
    ap.add_argument("--mode", default="fused", choices=["fused", "per_token"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prefill", action="store_true", help="skip the context-prefill leg (configs[3], N = 1 only)")
    ap.add_argument("--profile-steps", type=int, default=5)
    ap.add_argument("--discrete", action="store_true", help="discrete-action head (argmax over the first 18 logits)")
    ap.add_argument("--domains", default="metaworld", help="metaworld | dmcontrol | composuite | mimicgen | mixed")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --envs per GPU (default); strong: --envs is the JOB's env count, split env i -> rank i %% N "
                         "(BASELINE.json configs[4]: 256 Atari envs on 1/2/4/8 GPUs)")
    ap.add_argument("--gather-every", type=int, default=16,
                    help="N > 1: all-gather the action tokens of this many env steps in one collective (1 = per step)")
    ap.add_argument("--opt", action="append", default=[], metavar="NAME=VALUE",
                    help="xl_set_option passthrough for A/B runs, e.g. --opt microbatches=1 --opt state_impl=1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs and a seeded sample of the state as DIR/<name>.npy")
    args = ap.parse_args()
    _quiet_stdout()
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the CUDA path computed: not available with --impl reference")
        run_reference(args)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the xlstm_b200 path has no CPU fallback); "
                         "use --impl reference for the CPU arm")
    import torch.distributed as dist
    from lram_b200 import _lib as L
    from lram_b200.config import preset
    from lram_b200.engine import XLSTMEngine
    from lram_b200.rollout import OverlappedTokenGather, shard_env_ids
    from lram_b200.synth import make_state_dict, make_stream

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    cfg = preset(args.model)
    sd = make_state_dict(cfg, seed=0)
    if args.scaling == "strong":
        assert args.envs % world == 0, "--scaling strong needs --envs divisible by the GPU count"
        args.job_envs = args.envs
        args.envs = args.envs // world
    B = args.envs
    n_envs = B * world
    env_ids = shard_env_ids(n_envs, rank, world)
    K, W = args.steps, args.warmup
    mode = L.XL_MODE_FUSED if args.mode == "fused" else L.XL_MODE_PER_TOKEN
    flags = (0 if args.no_graph else L.XL_FLAG_GRAPH) | (L.XL_FLAG_DISCRETE if args.discrete else 0)

    eng = XLSTMEngine(cfg, sd, max_batch=B, device=dev)
    opts = {}
    for kv in args.opt:
        name, val = kv.split("=")
        eng.set_option(name, int(val))
        opts[name] = int(val)
    cache = eng.new_state(B)
    cache_nbytes = cache.nbytes()
    total = K + W
    n_stream = min(total, 64)                    # the synthetic stream is cycled; values don't affect timing
    states_np, rtg_np, _ = make_stream(cfg, env_ids, n_stream, domains=args.domains)
    d_states = torch.from_numpy(states_np).to(dev)      # resident in HBM before the timed region
    d_rtg = torch.from_numpy(rtg_np).to(dev)
    s_in = torch.empty(B, cfg.state_dim, device=dev)
    r_in = torch.empty(B, device=dev)
    out = {"action_tokens": torch.zeros(B, cfg.act_dim, dtype=torch.int32, device=dev),
           "action_preds": torch.zeros(B, cfg.act_dim, dtype=torch.float32, device=dev)}
    stream = torch.cuda.current_stream(dev)
    gatherer = OverlappedTokenGather(B, cfg.act_dim, world, dev, every=args.gather_every, engine=eng) \
        if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def dev_step(t):
        s_in.copy_(d_states[t % n_stream], non_blocking=True)
        r_in.copy_(d_rtg[t % n_stream], non_blocking=True)
        eng.policy_step(cache, s_in, r_in, mode=mode, flags=flags, out=out)
        if world > 1:
            return gatherer.submit(out["action_tokens"])     # NCCL all-gather on a side stream
        return out["action_tokens"]

    # ---------------- device-resident throughput ------------------------------------------------------------
    # nvidia-smi needs a few hundred ms to start (longer when 8 ranks start one each): start it before the warm-up
    sampler = ClockSampler(local_rank)
    sampler.start()
    for t in range(W):
        dev_step(t)
    barrier()
    eng.launch_count()
    sampler.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for t in range(W, W + K):
        dev_step(t)
    if gatherer is not None:
        gatherer.finish()                                    # the last gathers are inside the timed region
    ev1.record(stream)
    barrier()
    launches = eng.launch_count()
    ms_total = ev0.elapsed_time(ev1)
    if world > 1:
        tt = torch.tensor([ms_total], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total = tt.item()
    dumped = snapshot_outputs(cfg, out, cache) if args.dump_outputs and rank == 0 else None
    # A timed region shorter than ~1 s can fall between two nvidia-smi samples: keep the SAME steps running (untimed,
    # same count on every rank: derived from the all-reduced time) until the window under load is ~1.2 s long.
    extra = 0
    if ms_total < 1000.0:
        extra = int((1200.0 - ms_total) / max(ms_total / K, 1e-3))
        for t in range(W + K, W + K + extra):
            dev_step(t)
        if gatherer is not None:
            gatherer.finish()
        torch.cuda.synchronize(dev)
        barrier()
        eng.launch_count()
    clocks = sampler.stop()
    clocks["window"] = (f"the {K} timed steps + {extra} untimed steps of the same workload right after them"
                        if extra else f"the {K} timed steps")
    value = n_envs * K / (ms_total / 1e3)

    # ---------------- end to end through the host-buffer C-ABI call ------------------------------------------
    cache_e = eng.new_state(B)
    h_states = torch.from_numpy(states_np).pin_memory()
    h_rtg = torch.from_numpy(rtg_np).pin_memory()
    h_tok = torch.zeros(B, cfg.act_dim, dtype=torch.int32).pin_memory()
    h_act = torch.zeros(B, cfg.act_dim, dtype=torch.float32).pin_memory()
    g_tok = torch.zeros(B, cfg.act_dim, dtype=torch.int32, device=dev)

    h_s_in = torch.zeros(B, cfg.state_dim).pin_memory()     # the env-side buffers of the step: written by the host
    h_r_in = torch.zeros(B).pin_memory()                     # every step, read by the library every step

    def host_step(t):
        h_s_in.copy_(h_states[t % n_stream])                 # what an env does: put the new observation in place
        h_r_in.copy_(h_rtg[t % n_stream])
        eng.policy_step_host(cache_e, h_s_in, h_r_in, h_tok, h_act, mode=mode, flags=flags)
        if world > 1:
            gatherer.submit(g_tok)                # tokens are already in the ring (written by the step itself)

    for t in range(W):
        host_step(t)
    barrier()
    lat = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record(stream)
    for t in range(W, W + K):
        t0 = time.perf_counter()
        host_step(t)
        lat.append((time.perf_counter() - t0) * 1e3)
    if gatherer is not None:
        gatherer.finish()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    wall_ms = (time.perf_counter() - t_wall0) * 1e3
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), wall_ms)   # host wall clock of the same region (every step ends in a stream sync)
    if world > 1:
        tt = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_ms = tt.item()
    e2e_value = n_envs * K / (e2e_ms / 1e3)
    h2d = B * cfg.state_dim * 4 + B * 4
    d2h = B * cfg.act_dim * 4 * 2

    # ---------------- roofline of the state-step kernel (profiled replay, eager launches) --------------------
    peaks, peak_kind = measured_peaks()
    nh, dh = cfg.num_heads, cfg.head_dim
    alg_bytes = B * (8 * nh * dh * dh + 8 * nh * dh + 8 * nh)       # C, n, m read + write, per launch
    roof = None
    if rank == 0 and hasattr(eng.lib, "xl_profile_begin"):
        import ctypes as C
        eng.lib.xl_profile_begin(eng.handle)
        for t in range(args.profile_steps):
            s_in.copy_(d_states[t % n_stream])
            r_in.copy_(d_rtg[t % n_stream])
            eng.policy_step(cache, s_in, r_in, mode=mode, flags=flags & ~L.XL_FLAG_GRAPH, out=out)
        torch.cuda.synchronize(dev)
        ms_sum, cnt, step_ms = C.c_double(), C.c_int64(), C.c_double()
        eng.lib.xl_profile_end(eng.handle, C.byref(ms_sum), C.byref(cnt), C.byref(step_ms))
        if cnt.value:
            avg_ms = ms_sum.value / cnt.value
            # one launch covers the envs of one micro-batch (B envs when the step is not split)
            alg_bytes = alg_bytes * cfg.num_blocks * args.profile_steps // cnt.value
            ach = alg_bytes / (avg_ms / 1e3) / 1e9
            traffic, traffic_src = None, None
            for tname in ("r02_state_traffic.json", "r01_state_traffic.json"):
                tpath = os.path.join(ROOT, "profiles", tname)
                if traffic is None and os.path.exists(tpath):
                    with open(tpath) as fh:
                        rec = json.load(fh).get(f"{args.model}:{B}:impl{opts.get('state_impl', 1)}")
                    if rec and opts.get("microbatches", 1) == 1 and not opts.get("state_fuse"):
                        traffic = rec["traffic"]      # one ncu --set full capture of this kernel at this shape
                        traffic_src = f"static: ncu --set full capture recorded in profiles/{tname} (not measured in this run)"
            roof = {"bound": "hbm", "kernel": "mlstm_state_stream_tma_kernel", "achieved": ach,
                    "peak": peaks["hbm_gbs"], "peak_kind": peak_kind, "unit": "GB/s",
                    "frac": ach / peaks["hbm_gbs"], "traffic": traffic, "traffic_source": traffic_src,
                    "avg_launch_us": avg_ms * 1e3,
                    "launches_timed": cnt.value, "algorithmic_bytes_per_launch": alg_bytes,
                    # launches per env step x their average duration / the GRAPH-timed step of the headline number
                    "share_of_step": (cnt.value / args.profile_steps) * avg_ms / max(ms_total / K, 1e-9),
                    "share_of_step_basis": "per-launch CUDA-event time (eager replay) x launches per step / graph-timed "
                                           "ms_per_step"}
    if world > 1:
        dist.barrier()

    # ---------------- whole-step roofline: every block's state once + the weights, over the graph-timed step ----
    state_bytes_step = B * sum(cfg.algorithmic_bytes_per_env_layer_tokenstep() for i in range(cfg.num_blocks)
                               if not cfg.is_slstm(i))
    weight_bytes = 2 * cfg.encoder_params()
    step_s = ms_total / K / 1e3
    whole = {"algorithmic_bytes_per_step": state_bytes_step + weight_bytes,
             "achieved": (state_bytes_step + weight_bytes) / step_s / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
             "frac": (state_bytes_step + weight_bytes) / step_s / 1e9 / peaks["hbm_gbs"],
             "note": "fused 3-token step: C/n/m/conv of every block read + written once per env step (SURVEY.md §8d "
                     "per-unit bytes x B x L) + bf16 encoder weights once; divided by ms_per_step of `value`"}

    # ---------------- reference on this GPU, eager (rank 0, N == 1 only) ---------------------------------------
    gpu_eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        eng.close()
        del cache, cache_e
        torch.cuda.empty_cache()
        try:
            v, ms, timed = time_oracle(cfg, sd, B, 30, 3, os.cpu_count() or 1, budget_s=30, domains=args.domains,
                                       discrete=args.discrete, device="cuda")
            gpu_eager = {"value": v, "unit": UNIT, "ms_per_step": statistics.mean(ms), "steps": timed, "envs": B,
                         "what": "the oracle's op sequence (restated xlstm native PyTorch backend + LRAM embed/head), "
                                 "fp32, run eagerly on this GPU through PyTorch/cuBLAS: token-by-token block stack, "
                                 "one D2H read of the action per step"}
        except RuntimeError as ex:          # e.g. out of memory at the largest shards: report, do not fail the bench
            gpu_eager = {"unavailable": str(ex).splitlines()[0][:200]}
        torch.cuda.empty_cache()

    # ---------------- context prefill, BASELINE.json configs[3] (rank 0, N == 1 only) -----------------------------
    prefill = None
    if rank == 0 and world == 1 and not args.no_prefill and not args.no_cpu_baseline:
        try:
            prefill = prefill_leg(peaks)
        except RuntimeError as ex:
            prefill = {"unavailable": str(ex).splitlines()[0][:200]}
        torch.cuda.empty_cache()

    # ---------------- CPU baseline (rank 0, N == 1 only) ------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        b_cpu = cpu_sample(B)
        v, ms, timed = time_oracle(cfg, sd, b_cpu, 1000, 2, cores, budget_s=20, domains=args.domains,
                                   discrete=args.discrete)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{b_cpu} of {B} envs x {timed} env steps (~20 s), oracle port of the xlstm native "
                         f"PyTorch backend, fp32, {cores} threads (same sample definition as --impl reference)",
               "p50_ms_per_step": statistics.median(ms)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(args, world),
                           step_mode=args.mode, cuda_graph=not args.no_graph, options=opts,
                           weights="bf16 GEMM matrices", state="fp32", parallelism=f"env-sharded x{world}",
                           gather=(f"one NCCL all_gather of int32 action tokens per {args.gather_every} env steps, side "
                                   "stream, straight from the token ring the argmax kernel fills inside the graph")
                           if world > 1 else "none (1 GPU)",
                           l2=(f"state stream {cache_nbytes / 2**20:.0f} MiB per step exceeds the 126 MB L2"
                               if cache_nbytes > 126e6 else
                               f"state {cache_nbytes / 2**20:.0f} MiB fits in the 126 MB L2 and is NOT flushed between "
                               "steps (a resident state cache is this workload's steady state; latency-bound case)"),
                           l2_prefetch=("library default: 48 MiB of the next block's C warmed into L2 on a side stream "
                                        "while the current block's chain runs, when a block's C is 100-300 MB")
                           if "l2_prefetch_mb" not in opts else f"{opts['l2_prefetch_mb']} MiB (forced)"),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / K, "p50_ms": statistics.median(lat),
                    "p90_ms": sorted(lat)[int(0.9 * (len(lat) - 1))]},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "whole_step": whole,
            "cpu_baseline": cpu,
            "gpu_eager_baseline": gpu_eager,
            "context_prefill": prefill,
        }
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumped.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a.cpu().numpy())
        _emit(line)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
