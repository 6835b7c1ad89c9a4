"""CPU tests: the C-ABI library loads and exports every declared symbol; host-side logic (config, synth,
sharding, gather over gloo with world_size 2, checkpoint-prefix stripping). No compute calls without a GPU."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from lram_b200 import _lib as L
from lram_b200.config import preset
from lram_b200.rollout import shard_env_ids
from lram_b200.synth import SyntheticEnvBatch, is_bf16_weight, make_state_dict, make_stream

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    lib = L.load()
    syms = L.declared_symbols()
    assert len(syms) >= 14 and "xl_policy_step" in syms and "xl_mlstm_cell_step" in syms
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/xlstm_b200.h but not exported"
    assert lib.xl_abi_version() == L.XL_ABI_VERSION == 3


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback_fails_loudly():
    lib = L.load()
    cfg = preset("toy")
    c = L.XLConfig(embedding_dim=cfg.d, num_blocks=cfg.num_blocks, num_heads=cfg.num_heads, inner_dim=cfg.inner,
                   conv_kernel=4, qkv_blocksize=4, state_dim=204, act_dim=8, action_channels=256,
                   discrete_actions=18, tokens_per_step=3, action_token_pos=1, max_batch=2, ln_eps=1e-5,
                   cell_eps=1e-6, embed_ln_eps=1e-5, tok_min_val=-1.0, tok_max_val=1.0)
    h = C.c_void_p()
    rc = lib.xl_create(C.byref(c), C.byref(h))
    assert rc == L.XL_ERR_NO_DEVICE and not h.value
    assert b"no CPU fallback" in lib.xl_last_error()
    from lram_b200.engine import XLSTMEngine
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        XLSTMEngine(cfg, make_state_dict(cfg), max_batch=1)


def test_create_rejects_bad_config():
    lib = L.load()
    c = L.XLConfig(embedding_dim=65, num_blocks=1, num_heads=4, inner_dim=128, conv_kernel=4, qkv_blocksize=4,
                   state_dim=204, act_dim=8, action_channels=256, discrete_actions=18, tokens_per_step=3,
                   action_token_pos=1, max_batch=1, ln_eps=1e-5, cell_eps=1e-6, embed_ln_eps=1e-5,
                   tok_min_val=-1.0, tok_max_val=1.0)
    h = C.c_void_p()
    assert lib.xl_create(C.byref(c), C.byref(h)) == L.XL_ERR_UNSUPPORTED
    assert lib.xl_create(None, C.byref(h)) == L.XL_ERR_INVALID_ARG


def test_presets_and_bytes():
    c = preset("48M")
    assert (c.inner, c.head_dim, c.num_blocks) == (1536, 384, 12)
    assert c.head_out == 2192 and c.num_actions == 274
    assert preset("206M").state_bytes_per_env() > 120 * 2 ** 20


def test_synth_is_deterministic_and_sharded_streams_match():
    cfg = preset("toy")
    a = make_state_dict(cfg, seed=0)
    b = make_state_dict(cfg, seed=0)
    assert all(torch.equal(a[k], b[k]) for k in a)
    for k, v in a.items():
        if is_bf16_weight(k):
            assert torch.equal(v, v.to(torch.bfloat16).float())        # exactly representable in bf16
    full, rtg, _ = make_stream(cfg, range(6), 5, domains="mixed")
    part, rtg_p, _ = make_stream(cfg, [1, 3, 5], 5, domains="mixed")
    assert np.array_equal(full[:, [1, 3, 5]], part) and np.array_equal(rtg[:, [1, 3, 5]], rtg_p)
    envs = SyntheticEnvBatch(cfg, range(2), ep_len=3)
    envs.reset()
    dones = [envs.step(None)[2].copy() for _ in range(6)]
    assert [d.all() for d in dones] == [False, False, True, False, False, True]


def test_shard_rule_matches_reference():
    # custom_eval_callback.py:385: idx % world_size == rank
    assert shard_env_ids(10, 1, 4) == [1, 5, 9]
    allv = sorted(sum((shard_env_ids(10, r, 4) for r in range(4)), []))
    assert allv == list(range(10))


def test_strip_checkpoint_prefixes():
    from lram_b200.engine import strip_checkpoint_prefixes
    sd = {"module._orig_mod.encoder.layers.post_blocks_norm.weight": torch.zeros(1), "_orig_mod.embed_ln.bias": torch.ones(1)}
    out = strip_checkpoint_prefixes(sd)
    assert set(out) == {"encoder.layers.post_blocks_norm.weight", "embed_ln.bias"}


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from lram_b200.rollout import gather_env_results, shard_env_ids
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
n_envs = 7                                   # ragged shards: 4 + 3
ids = shard_env_ids(n_envs, rank, world)
local = torch.tensor([[e * 10 + j for j in range(8)] for e in ids], dtype=torch.int32)
full = gather_env_results(local, n_envs, rank, world)
want = torch.tensor([[e * 10 + j for j in range(8)] for e in range(n_envs)], dtype=torch.int32)
assert torch.equal(full, want), (rank, full)
ret = gather_env_results(torch.tensor([float(e) for e in ids]), n_envs, rank, world)
assert torch.equal(ret, torch.arange(n_envs, dtype=torch.float32))
# batched / deferred token gather: 7 steps, flush every 3 (two full rings + a partial one at finish())
from lram_b200.rollout import OverlappedTokenGather
B_local, A, steps = 4, 8, 7
for every in (1, 3, 16):
    g = OverlappedTokenGather(B_local, A, world, "cpu", every=every, keep=True)
    def tok(r, t):
        return torch.tensor([[1000 * t + 10 * (b * world + r) + j for j in range(A)] for b in range(B_local)],
                            dtype=torch.int32)
    for t in range(steps):
        g.submit(tok(rank, t))
    g.finish()
    assert g.flushes == -(-steps // every), (every, g.flushes)
    allsteps = torch.cat([g.global_view(r) for r in g.results], dim=0)        # [steps, n_envs, A]
    want = torch.stack([torch.tensor([[1000 * t + 10 * e + j for j in range(A)] for e in range(B_local * world)],
                                     dtype=torch.int32) for t in range(steps)])
    assert torch.equal(allsteps, want), (rank, every)
dist.barrier(); dist.destroy_process_group()
print("ok", rank)
"""


def test_gather_world_size_2_gloo(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(_GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29653", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script), ROOT], env=dict(env, RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_bench_reference_arm_prints_one_json_line_with_the_contract_keys():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): exactly ONE line on stdout, valid JSON, with
    the keys of the bench contract. Runs the oracle port on a toy-sized sample (no GPU)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--model", "16M",
                        "--envs", "1", "--steps", "2", "--warmup", "3"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["gpu_launches"] == 0 and d["steps"] == 2
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] and "model" in d["config"]


@pytest.mark.gpu
def test_bench_dump_outputs_equal_an_independent_run(tmp_path):
    """`bench.py --dump-outputs DIR` on a toy workload writes exactly what an engine stepped warmup + steps times over the
    same seeded stream holds after its last step (float32 / float64, under 64 MB), and one more step changes it."""
    import json
    import bench
    from lram_b200.engine import XLSTMEngine
    W, K, B = 3, 5, 4
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--model", "toy128", "--envs", str(B),
                        "--steps", str(K), "--warmup", str(W), "--no-cpu-baseline", "--profile-steps", "0",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == K
    got = {f.stem: np.load(f) for f in sorted(tmp_path.glob("*.npy"))}
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert sum(v.nbytes for v in got.values()) <= 64 * 2 ** 20

    cfg = preset("toy128")
    states, rtg, _ = make_stream(cfg, range(B), W + K, domains="metaworld")
    eng = XLSTMEngine(cfg, make_state_dict(cfg, seed=0), max_batch=B)
    cache = eng.new_state(B)
    s_in, r_in = torch.empty(B, cfg.state_dim, device="cuda"), torch.empty(B, device="cuda")
    out = {"action_tokens": torch.zeros(B, cfg.act_dim, dtype=torch.int32, device="cuda"),
           "action_preds": torch.zeros(B, cfg.act_dim, dtype=torch.float32, device="cuda")}

    def step(t):
        s_in.copy_(torch.from_numpy(states[t % (W + K)]))
        r_in.copy_(torch.from_numpy(rtg[t % (W + K)]))
        eng.policy_step(cache, s_in, r_in, mode=L.XL_MODE_FUSED, flags=L.XL_FLAG_GRAPH, out=out)

    for t in range(W + K):
        step(t)
    want = {k: v.cpu().numpy() for k, v in bench.snapshot_outputs(cfg, out, cache).items()}
    assert got.keys() == want.keys() and {"action_tokens", "action_preds", "state_block00_C"} <= set(got)
    for k in want:
        assert np.array_equal(got[k], want[k]), k
    assert got["action_tokens"].any() and got["state_block00_C"].any()
    step(W + K)
    later = bench.snapshot_outputs(cfg, out, cache)
    assert not np.array_equal(got["state_block00_C"], later["state_block00_C"].cpu().numpy())
    eng.close()


def test_every_option_of_the_library_is_documented_in_the_header():
    """xl_set_option names accepted by lram_b200/csrc/xl_api.cu must all be described in include/xlstm_b200.h (the header is
    the boundary a maintainer reads)."""
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    api = open(os.path.join(root, "lram_b200", "csrc", "xl_api.cu")).read()
    hdr = open(os.path.join(root, "include", "xlstm_b200.h")).read()
    body = api[api.index("int xl_set_option"):]
    names = sorted(set(re.findall(r'!strcmp\(name, "([a-z0-9_]+)"\)', body)))
    assert len(names) > 30
    missing = [n for n in names if f'"{n}"' not in hdr]
    assert not missing, missing
