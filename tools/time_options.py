"""Times the graph-replayed policy step under xl_set_option combinations WITHOUT checking equality (use tools/ab_options.py
for that): for experimental options whose results are under investigation.   python tools/time_options.py 206M:128 "state_fuse=2" ..."""
import json, os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lram_b200 import _lib as L
from lram_b200.config import preset
from lram_b200.engine import XLSTMEngine
from lram_b200.synth import make_state_dict, make_stream

name, B = sys.argv[1].split(":")
B = int(B)
steps = int(os.environ.get("AB_STEPS", "50"))
cfg = preset(name)
sd = make_state_dict(cfg, seed=0)
states, rtg, _ = make_stream(cfg, range(B), 2, domains="mixed")
for combo in sys.argv[2:]:
    eng = XLSTMEngine(cfg, sd, max_batch=B)
    for kv in combo.split(","):
        if kv:
            k, v = kv.split("=")
            eng.set_option(k, int(v))
    cache = eng.new_state(B)
    s_dev, r_dev = torch.from_numpy(states[0]).cuda(), torch.from_numpy(rtg[0]).cuda()
    out = None
    for _ in range(8):
        out = eng.policy_step(cache, s_dev, r_dev, flags=L.XL_FLAG_GRAPH, out=out)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            eng.policy_step(cache, s_dev, r_dev, flags=L.XL_FLAG_GRAPH, out=out)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / steps)
    print(json.dumps({"model": name, "B": B, "options": combo, "ms_per_step": round(best, 4),
                      "env_steps_per_s": round(B / best * 1e3, 1)}), flush=True)
    eng.close()
