"""Sequence forward of the policy (xl_policy_forward) against the prefill it extends, and against stepping.

    python tools/bench_policy_forward.py [--reps 3] [--out profiles/r05_policy_forward.json]

Workloads (policy form, seeded synthetic trajectories, rewards given):
  * 48M x 64 envs x Tn = 1024 timesteps;
  * 206M x 1 env x Tn = 16 666 timesteps (~50 k tokens: the longest context of BASELINE configs[3]).
Three calls alternate within every repetition, each from the same start state:
  prefill  : xl_policy_prefill (state only, no action outputs);
  fwd_lp   : xl_policy_forward with tokens + actions + log-probabilities of given targets;
  fwd_all  : the same plus the fp32 logits of every timestep.
Rates are timesteps per second (B * Tn over the call time). Graph-replayed stepping (xl_policy_step, XL_FLAG_GRAPH) is
timed at 48M x 64 envs for comparison. The working sets (the 48M x 64 recurrent state is 1.8 GB, the 206M weights
0.4 GB) exceed the 126 MB L2. Times are CUDA events around whole calls (each arm resets the state first) after one warm-up
call of every kind (workspaces grown); the forward arms call the library directly, outputs allocated beforehand. The card's name and power limit are read in the same run. GPU only.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from lram_b200 import _lib as L  # noqa: E402
from lram_b200.config import preset  # noqa: E402
from lram_b200.engine import XLSTMEngine  # noqa: E402
from lram_b200.synth import make_state_dict  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--step-iters", type=int, default=200)
ap.add_argument("--out", default="profiles/r05_policy_forward.json")
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_policy_forward.py measures on a GPU; none is visible")


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


def inputs(cfg, B, Tn, seed):
    g = torch.Generator("cuda").manual_seed(seed)
    states = torch.randn(B, Tn, cfg.state_dim, device="cuda", generator=g)
    rtg = torch.rand(B, Tn, device="cuda", generator=g)
    rew = torch.randn(B, Tn, device="cuda", generator=g) * 0.1
    tg = torch.randint(0, cfg.num_actions, (B, Tn, cfg.act_dim), device="cuda", generator=g)
    return states, rtg, rew, tg


def compare(model, B, Tn, reps):
    cfg = preset(model)
    eng = XLSTMEngine(cfg, make_state_dict(cfg, seed=0), max_batch=B)
    states, rtg, rew, tg = inputs(cfg, B, Tn, 1)
    st = eng.new_state(B)

    def prefill():
        eng.reset(st)
        eng.policy_prefill(st, states, rtg, rew)

    # the forward arms call the library directly with outputs allocated and targets checked once, outside the timed
    # window, so that every arm times the library call alone
    tg32 = tg.to(torch.int32).contiguous()
    tok = torch.empty(B, Tn, cfg.act_dim, dtype=torch.int32, device="cuda")
    act = torch.empty(B, Tn, cfg.act_dim, device="cuda")
    lp = torch.empty(B, Tn, cfg.act_dim, device="cuda")
    lg = torch.empty(B, Tn, cfg.head_out, device="cuda")

    def forward(logits):
        so = L.XLSeqOutputs(tokens=tok.data_ptr(), actions=act.data_ptr(), logits=lg.data_ptr() if logits else None,
                            targets=tg32.data_ptr(), logprobs=lp.data_ptr())
        eng.reset(st)
        L.check(eng.lib.xl_policy_forward(eng.handle, st.buf.data_ptr(), states.data_ptr(), rtg.data_ptr(),
                                          rew.data_ptr(), None, B, Tn, C.byref(so), 0,
                                          torch.cuda.current_stream().cuda_stream))

    def fwd_lp():
        forward(False)

    def fwd_all():
        forward(True)

    fns = (("prefill", prefill), ("fwd_lp", fwd_lp), ("fwd_all", fwd_all))
    for _, fn in fns:                                   # warm-up: workspaces grown, modules loaded
        fn()
    times = {k: [] for k, _ in fns}
    for _ in range(reps):
        for k, fn in fns:
            times[k].append(timed(fn))
    res = {"model": model, "envs": B, "Tn": Tn, "timesteps": B * Tn}
    for k, v in times.items():
        res[f"{k}_s"] = v
        res[f"{k}_timesteps_per_s"] = B * Tn / statistics.median(v)
    res["fwd_lp_over_prefill_time"] = statistics.median(times["fwd_lp"]) / statistics.median(times["prefill"])
    res["fwd_all_over_prefill_time"] = statistics.median(times["fwd_all"]) / statistics.median(times["prefill"])
    eng.close()
    return res


def stepping(model, B, iters):
    cfg = preset(model)
    eng = XLSTMEngine(cfg, make_state_dict(cfg, seed=0), max_batch=B)
    states, rtg, rew, _ = inputs(cfg, B, 1, 2)
    s, r, w = states[:, 0].contiguous(), rtg[:, 0].contiguous(), rew[:, 0].contiguous()
    st = eng.new_state(B)
    out = {"action_tokens": torch.zeros(B, cfg.act_dim, dtype=torch.int32, device="cuda"),
           "action_preds": torch.zeros(B, cfg.act_dim, device="cuda")}

    def run():
        for _ in range(iters):
            eng.policy_step(st, s, r, w, flags=L.XL_FLAG_GRAPH, out=out)

    for _ in range(10):
        eng.policy_step(st, s, r, w, flags=L.XL_FLAG_GRAPH, out=out)
    t = [timed(run) for _ in range(3)]
    eng.close()
    return {"model": model, "envs": B, "steps": iters, "step_s": [x / iters for x in t],
            "timesteps_per_s": B * iters / statistics.median(t)}


out = {"card": card(), "reps": args.reps, "cases": []}
for model, B, Tn in (("48M", 64, 1024), ("206M", 1, 16666)):
    r = compare(model, B, Tn, args.reps)
    print(json.dumps(r), flush=True)
    out["cases"].append(r)
r = stepping("48M", 64, args.step_iters)
print(json.dumps(r), flush=True)
out["graph_stepping"] = r
out["card_after"] = card()
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
print(json.dumps({"card": out["card"]}))
