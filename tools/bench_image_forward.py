"""Image observations on the sequence path: the sequence forward from state embeddings (xl_policy_forward_embeds)
against stepping the same trajectories, against the raw-state forward, and frames end to end.

    python tools/bench_image_forward.py [--reps 3] [--out profiles/r06_image_forward.json]

Workloads (seeded synthetic trajectories, rewards given): 48M x 16 envs x Tn = 4096 timesteps and 206M x 1 env x
Tn = 16 384 timesteps. Per workload, in one run:
  fwd_embeds : xl_policy_forward_embeds (tokens + actions) on [B, Tn, d] state embeddings;
  fwd_raw    : xl_policy_forward on [B, Tn, state_dim] raw states, same shape (alternated with fwd_embeds);
  stepping   : the status quo for image envs, Tn graph-replayed xl_policy_step(XL_FLAG_STATE_EMBEDS) calls, each after
               a copy of the timestep's [B, d] embeddings into the graph's input buffer (one repetition);
  e2e        : uint8 frames [B, Tn, 3, 64, 64] resident on the GPU -> image_encoder.embed_frames (ImpalaCNN in PyTorch
               / cuDNN, slices of 2048 frames) -> xl_policy_forward_embeds, with the CNN's time shown on its own.
Rates are timesteps per second (B * Tn over the call time). Times are CUDA events around whole calls after one warm-up
of every kind (workspaces grown); every forward arm resets the state first. The card's name and power limit are read in
the same run. GPU only.
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
from lram_b200.image_encoder import ImpalaCNN, embed_frames, make_impala_state_dict, split_image_weights  # noqa: E402
from lram_b200.synth import make_state_dict  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--out", default="profiles/r06_image_forward.json")
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_image_forward.py measures on a GPU; none is visible")


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


def case(model, B, Tn, reps):
    cfg = preset(model)
    eng = XLSTMEngine(cfg, make_state_dict(cfg, seed=0), max_batch=B)
    cnn = ImpalaCNN((3, 64, 64), cfg.d).cuda().eval()
    cnn.load_state_dict(split_image_weights(make_impala_state_dict(cfg.d, (3, 64, 64), seed=1)))
    g = torch.Generator("cuda").manual_seed(1)
    frames = torch.randint(0, 256, (B, Tn, 3, 64, 64), dtype=torch.uint8, device="cuda", generator=g)
    emb = embed_frames(cnn, frames)
    states = torch.randn(B, Tn, cfg.state_dim, device="cuda", generator=g)
    rtg = torch.rand(B, Tn, device="cuda", generator=g)
    rew = torch.randn(B, Tn, device="cuda", generator=g) * 0.1
    st = eng.new_state(B)
    tok = torch.empty(B, Tn, cfg.act_dim, dtype=torch.int32, device="cuda")
    act = torch.empty(B, Tn, cfg.act_dim, device="cuda")
    so = L.XLSeqOutputs(tokens=tok.data_ptr(), actions=act.data_ptr(), logits=None, targets=None, logprobs=None)
    stream = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731

    def fwd(fn, x):
        eng.reset(st)
        L.check(fn(eng.handle, st.buf.data_ptr(), x.data_ptr(), rtg.data_ptr(), rew.data_ptr(), None, B, Tn,
                   C.byref(so), 0, stream()))

    def fwd_embeds():
        fwd(eng.lib.xl_policy_forward_embeds, emb)

    def fwd_raw():
        fwd(eng.lib.xl_policy_forward, states)

    # status quo: one graph-replayed embedding step per timestep, inputs copied into the graph's buffers
    io = {"s": torch.empty(B, cfg.d, device="cuda"), "r": torch.empty(B, device="cuda"),
          "w": torch.empty(B, device="cuda")}
    res = {"action_tokens": torch.zeros(B, cfg.act_dim, dtype=torch.int32, device="cuda"),
           "action_preds": torch.zeros(B, cfg.act_dim, device="cuda")}

    def stepping():
        eng.reset(st)
        for t in range(Tn):
            io["s"].copy_(emb[:, t])
            io["r"].copy_(rtg[:, t])
            io["w"].copy_(rew[:, t])
            eng.policy_step(st, io["s"], io["r"], io["w"], flags=L.XL_FLAG_GRAPH, out=res, state_embeds=True)

    # warm-up of every kind; e2e = the CNN's time + the embeddings forward's time
    fwd_embeds()
    fwd_raw()
    for t in range(3):
        eng.policy_step(st, emb[:, t].contiguous(), rtg[:, t].contiguous(), rew[:, t].contiguous(),
                        flags=L.XL_FLAG_GRAPH, out=res, state_embeds=True)
    embed_frames(cnn, frames[:, :64], max_frames=2048)
    times = {"fwd_embeds": [], "fwd_raw": [], "cnn": []}
    for _ in range(reps):
        times["fwd_embeds"].append(timed(fwd_embeds))
        times["fwd_raw"].append(timed(fwd_raw))
        times["cnn"].append(timed(lambda: embed_frames(cnn, frames, max_frames=2048)))
    step_s = timed(stepping)
    ts = B * Tn
    med = {k: statistics.median(v) for k, v in times.items()}
    r = {"model": model, "envs": B, "Tn": Tn, "timesteps": ts}
    for k, v in times.items():
        r[f"{k}_s"] = v
        r[f"{k}_timesteps_per_s"] = ts / med[k]
    r["stepping_s"] = step_s
    r["stepping_timesteps_per_s"] = ts / step_s
    r["fwd_embeds_speedup_over_stepping"] = step_s / med["fwd_embeds"]
    r["fwd_embeds_over_fwd_raw_time"] = med["fwd_embeds"] / med["fwd_raw"]
    r["e2e_s"] = med["cnn"] + med["fwd_embeds"]
    r["e2e_timesteps_per_s"] = ts / r["e2e_s"]
    r["e2e_cnn_share"] = med["cnn"] / r["e2e_s"]
    # outputs agree: the forward's tokens against the last stepped timestep
    fwd_embeds()
    torch.cuda.synchronize()
    r["last_step_tokens_equal_forward"] = bool(torch.equal(tok[:, -1], res["action_tokens"]))
    eng.close()
    del frames, emb, states
    torch.cuda.empty_cache()
    return r


out = {"card": card(), "reps": args.reps, "cases": []}
for model, B, Tn in (("48M", 16, 4096), ("206M", 1, 16384)):
    r = case(model, B, Tn, args.reps)
    print(json.dumps(r), flush=True)
    out["cases"].append(r)
out["card_after"] = card()
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
print(json.dumps({"card": out["card"]}))
