"""Ragged context prefill (xl_prefill_ragged): one call with a context length per env, against the two ways of doing
the same job without it, and the cost of its state gather / scatter.

    python tools/bench_ragged_prefill.py [--tokens 50000] [--reps 2] [--out profiles/r04_ragged_prefill.json]

Cases (encoder form, embedded tokens, no hidden-state output; seeded lengths uniform in [S/8, S]):
  * 206M x 8 envs and 48M x 64 envs, three ways, alternated within each repetition:
      ragged   : one xl_prefill_ragged call;
      separate : B prefills of one env each (xl_prefill at B = 1, S = that env's length), back to back;
      padded   : one uniform xl_prefill of all envs over max(lengths) tokens. This leaves the WRONG state (every token
                 moves the state); it is timed only as a cost reference.
    Rates count real tokens only (sum of lengths) for all three.
  * 48M, one active env among 64 (not env 0, so its slot goes through the state gather / scatter) against a B = 1
    prefill of the same S/8 tokens. The gap is the gather + scatter of one env's state only when S/8 is a multiple of
    16: otherwise the B = 1 call steps its remainder through the step path and the gap also holds that difference (the
    script then reports no GB/s for a negative gap).
Times are CUDA events around whole calls after a warm-up call of every shape (workspaces grown). The card's name and
power limit are read in the same run. GPU only.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from lram_b200.config import preset  # noqa: E402
from lram_b200.engine import XLSTMEngine  # noqa: E402
from lram_b200.synth import make_state_dict  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--tokens", type=int, default=50000, help="S: longest context (tokens)")
ap.add_argument("--reps", type=int, default=2)
ap.add_argument("--seed", type=int, default=0)
ap.add_argument("--out", default="profiles/r04_ragged_prefill.json")
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_ragged_prefill.py measures on a GPU; none is visible")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    first = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": first}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3


def compare(model, B, S, reps, rng):
    cfg = preset(model)
    eng = XLSTMEngine(cfg, make_state_dict(cfg, seed=0), max_batch=B)
    lengths = rng.integers(S // 8, S + 1, B).astype(np.int32)
    x = torch.randn(B, S, cfg.d, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    real = int(lengths.sum())
    st, st1 = eng.new_state(B), eng.new_state(1)

    def ragged():
        eng.prefill(st, x, want_hidden=False, lengths=lengths)

    def separate():
        for b in range(B):
            eng.prefill(st1, x[b:b + 1, :lengths[b]], want_hidden=False)

    xp = x[:, :int(lengths.max())].contiguous()

    def padded():
        eng.prefill(st, xp, want_hidden=False)

    # warm-up: every shape once at a short context (chunk rows, compact state and cell workspaces as in the timed calls)
    w = min(S, 4096)
    eng.prefill(st, x[:, :w], want_hidden=False, lengths=np.maximum(lengths * w // S, 1))
    eng.prefill(st1, x[:1, :min(S, 20000)], want_hidden=False)
    eng.prefill(st, x[:, :w], want_hidden=False)
    times = {"ragged": [], "separate": [], "padded": []}
    for _ in range(reps):
        for k, fn in (("ragged", ragged), ("separate", separate), ("padded", padded)):
            times[k].append(timed(fn))
    res = {"model": model, "envs": B, "S": S, "lengths_min": int(lengths.min()), "lengths_max": int(lengths.max()),
           "real_tokens": real, "padded_tokens": int(lengths.max()) * B}
    for k, v in times.items():
        res[f"{k}_s"] = v
        res[f"{k}_real_tokens_per_s"] = real / statistics.median(v)
    res["ragged_speedup_vs_separate"] = statistics.median(times["separate"]) / statistics.median(times["ragged"])
    res["ragged_speedup_vs_padded"] = statistics.median(times["padded"]) / statistics.median(times["ragged"])
    eng.close()
    return res


def one_active(model, B, S, reps):
    cfg = preset(model)
    eng = XLSTMEngine(cfg, make_state_dict(cfg, seed=0), max_batch=B)
    env = B // 2 + 5
    lengths = np.zeros(B, np.int32)
    lengths[env] = S
    x = torch.randn(B, S, cfg.d, device="cuda", generator=torch.Generator("cuda").manual_seed(2))
    st, st1 = eng.new_state(B), eng.new_state(1)
    x1 = x[env:env + 1].contiguous()

    def ragged():
        eng.prefill(st, x, want_hidden=False, lengths=lengths)

    def single():
        eng.prefill(st1, x1, want_hidden=False)

    ragged()
    single()
    t_r, t_1 = [], []
    for _ in range(reps * 3):
        t_r.append(timed(ragged))
        t_1.append(timed(single))
    env_bytes = int(eng.lib.xl_state_bytes(eng.handle, 1))
    gap = statistics.median(t_r) - statistics.median(t_1)
    moved = 4 * env_bytes          # gather: read + write one slot; scatter: the same
    res = {"model": model, "envs": B, "active_env": env, "S": S, "ragged_s": t_r, "single_env_prefill_s": t_1,
           "gap_s": gap, "env_state_bytes": env_bytes, "gather_scatter_bytes": moved,
           "gather_scatter_GBps_over_gap": moved / gap / 1e9 if gap > 0 else None}
    eng.close()
    return res


rng = np.random.default_rng(args.seed)
out = {"card": card(), "S": args.tokens, "reps": args.reps, "cases": []}
for model, B in (("206M", 8), ("48M", 64)):
    r = compare(model, B, args.tokens, args.reps, rng)
    print(json.dumps(r), flush=True)
    out["cases"].append(r)
r = one_active("48M", 64, args.tokens // 8, args.reps)
print(json.dumps(r), flush=True)
out["one_active"] = r
out["card_after"] = card()
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
print(json.dumps({"card": out["card"]}))
