"""Cost of the device sampler (xl_set_sampling) on the graph-replayed policy step.

    python tools/bench_sampling.py [--steps 200] [--reps 4] [--out profiles/sampling.json]

Per config: argmax and sampled steps (default `a_sample_kwargs`: temperature 1, top_p 0.5, top_k 0) alternate in blocks
of `steps` within one run, each timed with CUDA events around the block; the eager torch tail (`policy_step` with logits
+ `sample_from_logits` + the host read of the tokens) is timed the same way; then `BatchedRollout` env-steps/s with the
sampler armed. Prints the card name and power limit beside the numbers and writes them as JSON to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from lram_b200 import _lib as L  # noqa: E402
from lram_b200.config import preset  # noqa: E402
from lram_b200.decision_xlstm import sample_from_logits  # noqa: E402
from lram_b200.engine import XLSTMEngine  # noqa: E402
from lram_b200.rollout import BatchedRollout  # noqa: E402
from lram_b200.synth import SyntheticEnvBatch, make_state_dict, make_stream  # noqa: E402

KW = dict(temperature=1.0, top_k=0, top_p=0.5)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def bench_config(name, B, discrete, steps, reps):
    cfg = preset(name)
    eng = XLSTMEngine(cfg, make_state_dict(cfg, seed=0), max_batch=B)
    states, rtg, _ = make_stream(cfg, range(B), 1)
    s_dev, r_dev = torch.from_numpy(states[0]).cuda(), torch.from_numpy(rtg[0]).cuda()
    flags = (L.XL_FLAG_DISCRETE if discrete else 0) | L.XL_FLAG_GRAPH
    cache = eng.new_state(B)
    out = eng.policy_step(cache, s_dev, r_dev, flags=flags)

    def step():
        eng.policy_step(cache, s_dev, r_dev, flags=flags, out=out)

    res = {"argmax": [], "sampled": []}
    for kind in ("argmax", "sampled"):               # warm both graphs
        eng.set_sampling(**KW, seed=1) if kind == "sampled" else eng.set_sampling(None)
        timed(step, 20)
    for _ in range(reps):
        for kind in ("argmax", "sampled"):
            eng.set_sampling(**KW, seed=1) if kind == "sampled" else eng.set_sampling(None)
            timed(step, 3)                          # arming / disarming drops the graph: re-capture outside the window
            res[kind].append(timed(step, steps))
    eng.set_sampling(None)
    R = 1 if discrete else cfg.act_dim
    eager_out = eng.policy_step(cache, s_dev, r_dev, flags=flags & ~L.XL_FLAG_GRAPH, want_logits=True)

    def torch_tail():
        o = eng.policy_step(cache, s_dev, r_dev, flags=flags & ~L.XL_FLAG_GRAPH, want_logits=True, out=eager_out)
        sample_from_logits(o["action_logits"].view(B, R, cfg.num_actions), **KW).cpu()

    timed(torch_tail, 5)
    tail = timed(torch_tail, max(20, steps // 4))
    eng.close()
    a, s = statistics.median(res["argmax"]), statistics.median(res["sampled"])
    return {"config": f"{name} x {B} {'discrete' if discrete else 'continuous'}", "argmax_ms": a, "sampled_ms": s,
            "sampled_over_argmax": s / a - 1.0, "argmax_ms_blocks": res["argmax"], "sampled_ms_blocks": res["sampled"],
            "steps_per_block": steps, "eager_torch_tail_ms": tail}


def bench_rollout(name, B, n_steps):
    cfg = preset(name)
    eng = XLSTMEngine(cfg, make_state_dict(cfg, seed=0), max_batch=B)
    out = {}
    for kind, kw in (("argmax", None), ("sampled", KW)):
        ro = BatchedRollout(eng, SyntheticEnvBatch(cfg, range(B), ep_len=10 ** 9), sample_kwargs=kw, seed=1)
        ro.run(10)
        t0 = time.perf_counter()
        r = ro.run(n_steps)
        out[f"{kind}_env_steps_per_s"] = r["env_steps"] / (time.perf_counter() - t0)
        eng.set_sampling(None)
    eng.close()
    return {"config": f"BatchedRollout {name} x {B}", **out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=4)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sampling.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    gpu = card()
    rows = [bench_config("48M", 64, False, a.steps, a.reps), bench_config("110M", 256, True, a.steps, a.reps),
            bench_rollout("48M", 64, 300)]
    for r in rows:
        print(json.dumps(r))
    print(f"card: {gpu}")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump({"card": gpu, "results": rows}, fh, indent=1)


if __name__ == "__main__":
    np.set_printoptions(precision=4)
    main()
