"""Device action sampling (xl_set_sampling / xl_sample_actions): the contract written at xl_set_sampling in
include/xlstm_b200.h, restated here on the host in fp64 numpy with a Python Philox4x32-10, and checked against
`sample_from_logits` (the reference's `a_sample_kwargs`) on the CPU and against the library on the GPU."""
import math

import numpy as np
import pytest
import torch

from lram_b200 import _lib as L
from lram_b200 import decision_xlstm as DX
from lram_b200.config import preset
from lram_b200.synth import make_state_dict, make_stream

gpu = pytest.mark.gpu
MASK = 0xFFFFFFFF


# ---- host reference ------------------------------------------------------------------------------------------------
def philox4x32_10(ctr, key):
    c, (k0, k1) = [int(v) & MASK for v in ctr], (int(key[0]) & MASK, int(key[1]) & MASK)
    for r in range(10):
        if r:
            k0, k1 = (k0 + 0x9E3779B9) & MASK, (k1 + 0xBB67AE85) & MASK
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [(p1 >> 32) ^ c[1] ^ k0, p1 & MASK, (p0 >> 32) ^ c[3] ^ k1, p0 & MASK]
    return c


def uniform(step, gid, j, seed):
    x = philox4x32_10((step, gid, j, 0), (seed & MASK, seed >> 32))
    return ((x[0] >> 5) * 2 ** 26 + (x[1] >> 6)) * 2.0 ** -53


def host_candidates(block, top_p, top_k):
    """block [E, R, n] (one env = R rows) -> bool [E, R, n]: the candidates the contract draws from, -inf excluded."""
    x = np.asarray(block, dtype=np.float32).astype(np.float64)
    E, R, n = x.shape
    keep = np.ones(x.shape, bool)
    tp = float(np.float32(top_p))
    if tp > 0:
        rank = tp * (n - 1)
        lo, hi = math.floor(rank), math.ceil(rank)
        w = rank - lo
        v = np.sort(x, -1)
        a, e = v[..., lo], v[..., hi]
        pct = a + w * (e - a) if w < 0.5 else e - (e - a) * (1.0 - w)
        with np.errstate(invalid="ignore"):
            guard = (pct != x.reshape(E, -1).max(-1)[:, None]).all(1)
            keep = np.where(guard[:, None, None], x > pct[..., None], True)
    m = np.where(keep, x, -np.inf)
    if top_k > 0:
        order = np.argsort(-m, axis=-1, kind="stable")          # descending, ties: lowest index first
        keep &= np.argsort(order, axis=-1) < top_k              # rank of each position
    return keep & (m > -np.inf)                                 # +inf stays: its row then has no finite max


def host_argmax(row, n):
    r = np.asarray(row[:n], np.float32)
    nan = np.nonzero(np.isnan(r))[0]
    return int(nan[0]) if len(nan) else int(np.argmax(r))


def host_sample(block, temperature, top_p, top_k, seed, step, gids, discrete_actions, discrete):
    """-> tokens [E, R], number of rows whose u*Z lies within 1e-12 Z of a partial-sum boundary."""
    x = np.asarray(block, dtype=np.float32).astype(np.float64)
    E, R, n = x.shape
    cand = host_candidates(block, top_p, top_k)
    T = float(np.float32(temperature))
    tok = np.zeros((E, R), np.int64)
    near = 0
    for e in range(E):
        for j in range(R):
            c = cand[e, j]
            row = x[e, j]
            lmax = row[c].max() if c.any() else -np.inf
            if np.isnan(row).any() or not np.isfinite(lmax):
                tok[e, j] = host_argmax(block[e, j], discrete_actions if discrete else n)
                continue
            w = np.where(c, np.exp(T * (row - lmax)), 0.0)
            cs = np.cumsum(w)
            Z = cs[-1]
            target = uniform(step, gids[e], j, seed) * Z
            hit = np.nonzero(cs > target)[0]
            tok[e, j] = hit[0] if len(hit) else np.nonzero(w > 0)[0][-1]
            near += bool((np.abs(cs[w > 0] - target) <= 1e-12 * Z).any())
    return tok, near


def host_probs(row, temperature, top_p, top_k):
    x = np.asarray(row, np.float32).astype(np.float64)
    c = host_candidates(x[None, None], top_p, top_k)[0, 0]
    w = np.where(c, np.exp(float(np.float32(temperature)) * (x - x[c].max())), 0.0)
    return w / w.sum()


def token_actions(tok, cfg, discrete):
    if discrete:
        return tok.astype(np.float32)
    bw = np.float32((1.0 - (-1.0)) / cfg.action_channels)
    return np.maximum(tok - cfg.discrete_actions, 0).astype(np.float32) * bw + np.float32(-1.0)


# ---- CPU -----------------------------------------------------------------------------------------------------------
def test_philox_known_answers():
    assert philox4x32_10((0, 0, 0, 0), (0, 0)) == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    assert philox4x32_10((MASK,) * 4, (MASK, MASK)) == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]


def _crafted_rows(n, rng):
    rows = []
    r = rng.standard_normal(n).astype(np.float32)
    r[[3, 70, 200]] = r.max() + 1.0                 # ties at the max
    rows.append(r)
    r = np.round(rng.standard_normal(n) * 2).astype(np.float32)   # many ties, incl. at the k-th value
    rows.append(r)
    r = np.zeros(n, np.float32)
    r[10:20] = 1.0                                  # a plateau of 10 equal maxima, k = 5 cuts inside it
    rows.append(r)
    return rows


def _sample_from_logits_cut(monkeypatch, logits, top_p, top_k):
    """The candidate set `sample_from_logits` hands to Categorical: its finite logits (mapped through topk indices)."""
    seen = {}

    class Rec:
        def __init__(self, logits):
            seen["logits"] = logits

        def sample(self):
            return torch.zeros(seen["logits"].shape[:-1], dtype=torch.long)

    orig_topk = torch.topk

    def topk(t, k):
        v, i = orig_topk(t, k)
        seen["idx"] = i
        return v, i

    monkeypatch.setattr(torch.distributions, "Categorical", Rec)
    monkeypatch.setattr(torch, "topk", topk)
    DX.sample_from_logits(torch.from_numpy(logits), temperature=1.0, top_k=top_k, top_p=top_p)
    monkeypatch.undo()
    fin = (seen["logits"] > -float("inf")).numpy()
    out = np.zeros(logits.shape, bool)
    if top_k > 0:
        np.put_along_axis(out, seen["idx"].numpy(), fin, -1)
    else:
        out = fin
    return out


@pytest.mark.parametrize("rows", [1, 8])
def test_host_cut_equals_sample_from_logits_cut(monkeypatch, rows):
    """The host reference's candidate set is the cut `sample_from_logits` makes, for one env's [1, 274] discrete row or
    [8, 274] continuous block, including ties at the max and at the k-th value. Where equal values straddle the top-k
    boundary, torch.topk leaves unspecified which of them it keeps (on the CPU it keeps e.g. 11, 13, 12, 14, 10 of a
    plateau at 10..19); the contract keeps the lowest indices. There the two sets hold the same values."""
    rng = np.random.default_rng(0)
    n = preset("toy128").num_actions
    blocks = [(rng.standard_normal((rows, n)) * 3).astype(np.float32) for _ in range(4)]
    crafted = _crafted_rows(n, rng)
    blocks += [np.stack([crafted[(i + k) % len(crafted)] for i in range(rows)]) for k in range(len(crafted))]
    for blk in blocks:
        for top_p in (0.0, 0.5, 0.9, 1.0):
            for top_k in (0, 1, 5, n):
                want = _sample_from_logits_cut(monkeypatch, blk, top_p, top_k)
                got = host_candidates(blk[None], top_p, top_k)[0]
                for j in range(rows):
                    assert np.array_equal(np.sort(blk[j][got[j]]), np.sort(blk[j][want[j]])), (rows, top_p, top_k, j)
                    kept = np.sort(blk[j][got[j]])
                    straddles = top_k and len(kept) == top_k and (blk[j][~got[j]] == kept[0]).any()
                    if not straddles:
                        assert np.array_equal(got[j], want[j]), (rows, top_p, top_k, j)


def test_set_sampling_rejects_invalid_parameters_before_any_device_call():
    from lram_b200.engine import XLSTMEngine, sampling_params
    cfg = preset("toy128")

    class NoLib:
        def __getattr__(self, name):
            raise AssertionError(f"{name} reached the library")

    eng = XLSTMEngine.__new__(XLSTMEngine)
    eng.cfg, eng.lib, eng.handle = cfg, NoLib(), None
    bad = [dict(temperature=0.0), dict(temperature=-1.0), dict(temperature=float("nan")), dict(temperature=float("inf")),
           dict(top_p=-0.1), dict(top_p=1.5), dict(top_p=float("nan")), dict(top_k=-1), dict(top_k=cfg.num_actions + 1),
           dict(env_id_base=-1), dict(env_id_stride=0), dict(seed=-1), dict(seed=2 ** 64)]
    for kw in bad:
        with pytest.raises(ValueError):
            eng.set_sampling(**kw)
        with pytest.raises(ValueError):
            sampling_params(cfg, **kw)
    with pytest.raises(ValueError):
        eng.set_sampling(step0=-1)
    p = sampling_params(cfg, temperature=0.7, top_k=cfg.num_actions, top_p=1.0, seed=2 ** 64 - 1)
    assert (p.top_k, p.seed) == (cfg.num_actions, 2 ** 64 - 1)


# ---- GPU -----------------------------------------------------------------------------------------------------------
def _engine(name, B, **over):
    from lram_b200.engine import XLSTMEngine
    cfg = preset(name, **over)
    return cfg, XLSTMEngine(cfg, make_state_dict(cfg, seed=0), max_batch=B)


def _blocks(logits, cfg, discrete):
    return logits.reshape(logits.shape[0], 1 if discrete else cfg.act_dim, cfg.num_actions)


@gpu
def test_exact_draws_equal_host_reference():
    cfg, eng = _engine("toy128", 256)
    n = cfg.num_actions
    rng = np.random.default_rng(1)
    near_total = 0
    for discrete in (True, False):
        R = 1 if discrete else cfg.act_dim
        lg = (rng.standard_normal((256, R, n)) * 3).astype(np.float32)
        lg[5, 0, 17] = np.nan                      # NaN row -> argmax
        lg[6, 0, :] = 0.5                          # all equal: the cut leaves nothing (when the guard passes)
        lg[7, 0, :] = -np.inf                      # no finite logit
        lg[8, 0, 3] = np.inf
        for k, r in enumerate(_crafted_rows(n, rng)):
            lg[9 + k, 0] = r
        dev = torch.from_numpy(lg.reshape(256, -1)).cuda()
        for top_p in (0.0, 0.5, 0.9, 1.0):
            for top_k in (0, 1, 5, n):
                for temperature, step, seed in ((1.0, 0, 0), (0.7, 12345, 2 ** 40 + 7), (1.3, 2 ** 32 - 1, 99)):
                    tok, act = eng.sample_actions(dev, step, temperature=temperature, top_k=top_k, top_p=top_p,
                                                  seed=seed, discrete=discrete)
                    want, near = host_sample(lg, temperature, top_p, top_k, seed, step, range(256),
                                             cfg.discrete_actions, discrete)
                    got = tok.cpu().numpy()[:, :R]
                    bad = int((got != want).sum())
                    near_total += near
                    assert bad <= near, (discrete, top_p, top_k, temperature, bad, near)
                    assert np.array_equal(act.cpu().numpy()[:, :R], token_actions(got, cfg, discrete))
    print(f"rows within 1e-12 Z of a partial-sum boundary: {near_total}")
    eng.close()


def _chisq_p(counts, probs, N):
    from scipy.stats import chisquare
    exp = probs * N
    big = exp >= 5
    obs = np.append(counts[big], counts[~big].sum())
    ex = np.append(exp[big], exp[~big].sum())
    if ex[-1] == 0:
        obs, ex = obs[:-1], ex[:-1]
    assert counts[probs == 0].sum() == 0
    return chisquare(obs, ex).pvalue


@gpu
def test_draw_distribution_chi_square():
    """2^17 draws of one fixed row (4096 envs x 32 steps) follow the exact candidate probabilities."""
    B, steps = 4096, 32
    cfg, eng = _engine("toy128", B)
    n = cfg.num_actions
    row = (np.random.default_rng(2).standard_normal(n) * 2).astype(np.float32)
    dev = torch.from_numpy(np.tile(row, (B, 1))).cuda()
    for temperature in (0.5, 1.0, 1.3):
        for top_p, top_k in ((0.0, 0), (0.5, 0), (0.0, 5), (0.9, 20)):
            toks = torch.cat([eng.sample_actions(dev, s, temperature=temperature, top_k=top_k, top_p=top_p, seed=11,
                                                 discrete=True)[0][:, 0] for s in range(steps)])
            counts = np.bincount(toks.cpu().numpy(), minlength=n)
            p = _chisq_p(counts, host_probs(row, temperature, top_p, top_k), B * steps)
            assert p > 1e-6, (temperature, top_p, top_k, p)
    tok = eng.sample_actions(dev, 0, temperature=1e4, top_p=0.0, seed=3, discrete=True)[0][:, 0]
    assert (tok.cpu().numpy() == int(np.argmax(row))).all()
    eng.close()


def _run_steps(eng, cfg, B, steps, flags, armed=None, want_logits=True, step0=0):
    states, rtg, _ = make_stream(cfg, range(B), steps)
    cache = eng.new_state(B)
    if armed is not None:
        eng.set_sampling(**armed, step0=step0)
    s_dev = torch.zeros(B, cfg.state_dim, device="cuda")
    r_dev = torch.zeros(B, device="cuda")
    out, res = None, []
    for t in range(steps):
        s_dev.copy_(torch.from_numpy(states[t]))
        r_dev.copy_(torch.from_numpy(rtg[t]))
        out = eng.policy_step(cache, s_dev, r_dev, flags=flags, want_logits=want_logits, out=out)
        torch.cuda.synchronize()
        res.append({k: v.cpu().clone() for k, v in out.items()})
    return res


KW = dict(temperature=1.0, top_k=0, top_p=0.5, seed=5)


@gpu
@pytest.mark.parametrize("name,B,discrete", [("16M", 1, False), ("48M", 64, False), ("110M", 256, True)])
def test_policy_step_samples_its_own_logits(name, B, discrete):
    cfg, eng = _engine(name, B)
    flags = L.XL_FLAG_DISCRETE if discrete else 0
    R = 1 if discrete else cfg.act_dim
    step0 = 40
    res = _run_steps(eng, cfg, B, 3, flags, armed=KW, step0=step0)
    for t, o in enumerate(res):
        lg = _blocks(o["action_logits"].numpy(), cfg, discrete)
        want, near = host_sample(lg, 1.0, 0.5, 0, 5, step0 + t, range(B), cfg.discrete_actions, discrete)
        got = o["action_tokens"].numpy()[:, :R]
        assert int((got != want).sum()) <= near, (t, near)
        assert np.array_equal(o["action_preds"].numpy()[:, :R], token_actions(got, cfg, discrete))
    # graph replay == eager; the host-buffer step == the device-buffer step
    graph = _run_steps(eng, cfg, B, 3, flags | L.XL_FLAG_GRAPH, armed=KW, step0=step0)
    for a, b in zip(res, graph):
        assert torch.equal(a["action_tokens"], b["action_tokens"])
    if B <= 64:
        states, rtg, _ = make_stream(cfg, range(B), 3)
        eng.set_sampling(**KW, step0=step0)
        cache = eng.new_state(B)
        h_s = torch.zeros(B, cfg.state_dim, pin_memory=True)
        h_r = torch.zeros(B, pin_memory=True)
        h_t = torch.zeros(B, cfg.act_dim, dtype=torch.int32, pin_memory=True)
        h_a = torch.zeros(B, cfg.act_dim, pin_memory=True)
        for t in range(3):
            h_s.copy_(torch.from_numpy(states[t]))
            h_r.copy_(torch.from_numpy(rtg[t]))
            eng.policy_step_host(cache, h_s, h_r, h_t, h_a, flags=flags | L.XL_FLAG_GRAPH)
            assert torch.equal(h_t, res[t]["action_tokens"])
    eng.close()


@gpu
def test_microbatched_step_samples_the_same_tokens():
    cfg, eng = _engine("16M", 40)
    from test_gpu_parity import _microbatches_enabled
    if not _microbatches_enabled(eng):
        eng.close()
        pytest.skip("env micro-batches are refused by this build")
    one = _run_steps(eng, cfg, 40, 3, 0, armed=KW)
    eng.set_option("microbatches", 2)
    two = _run_steps(eng, cfg, 40, 3, 0, armed=KW)
    for a, b in zip(one, two):
        assert torch.equal(a["action_tokens"], b["action_tokens"])
    eng.close()


@gpu
def test_sharded_draws_equal_single_gpu_draws():
    cfg, eng = _engine("toy128", 16)
    lg = torch.randn(16, cfg.head_out, generator=torch.Generator().manual_seed(4)).mul(3).cuda()
    kw = dict(temperature=0.8, top_k=5, top_p=0.5, seed=17)
    full = eng.sample_actions(lg, 9, **kw)[0]
    for r in (0, 1):
        part = eng.sample_actions(lg[r::2].contiguous(), 9, env_id_base=r, env_id_stride=2, **kw)[0]
        assert torch.equal(part, full[r::2])
    # policy level: a stride-2 engine (rank 1 of 2) draws with the global ids 1 + 2b
    res = _run_steps(eng, cfg, 8, 2, 0, armed=dict(KW, env_id_base=1, env_id_stride=2), step0=3)
    for t, o in enumerate(res):
        lg = _blocks(o["action_logits"].numpy(), cfg, False)
        want, near = host_sample(lg, 1.0, 0.5, 0, 5, 3 + t, [1 + 2 * b for b in range(8)], cfg.discrete_actions, False)
        assert int((o["action_tokens"].numpy() != want).sum()) <= near
    eng.close()


@gpu
def test_token_ring_holds_sampled_tokens():
    cfg, eng = _engine("toy128", 6)
    ring = torch.full((4, 6, cfg.act_dim), -1, dtype=torch.int32, device="cuda")
    eng.set_token_ring(ring, 0)
    res = _run_steps(eng, cfg, 6, 3, L.XL_FLAG_GRAPH, armed=dict(KW, top_p=0.0))
    for t, o in enumerate(res):
        assert torch.equal(ring[t].cpu(), o["action_tokens"])
    eng.set_token_ring(None)
    eng.close()


@gpu
def test_batched_rollout_sampling_is_seeded():
    from lram_b200.rollout import BatchedRollout
    from lram_b200.synth import SyntheticEnvBatch
    cfg, eng = _engine("toy128", 8)
    kw = dict(temperature=1.0, top_k=0, top_p=0.0)
    runs = []
    for seed in (1, 1, 2):
        ro = BatchedRollout(eng, SyntheticEnvBatch(cfg, range(8), ep_len=5), sample_kwargs=kw, seed=seed)
        runs.append(ro.run(12, record=True)["tokens"])
    assert np.array_equal(runs[0], runs[1])
    assert not np.array_equal(runs[0], runs[2])
    argmax = BatchedRollout(eng, SyntheticEnvBatch(cfg, range(8), ep_len=5))
    eng.set_sampling(None)
    assert not np.array_equal(argmax.run(12, record=True)["tokens"], runs[0])
    eng.close()


@gpu
def test_agent_device_sampling_through_custom_evaluate_policy():
    """`a_sample_kwargs` + `a_sample_seed`: the env receives the step's sampled tokens, each in its candidate set."""
    import os
    import sys
    from lram_b200.decision_xlstm import DiscreteDecisionXLSTM, MultiDomainDiscreteDecisionXLSTMModel
    from lram_b200.rollout import custom_evaluate_policy
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from ref_stubs import Box
    cfg = preset("toy128")
    policy = MultiDomainDiscreteDecisionXLSTMModel(cfg, make_state_dict(cfg, seed=5), max_batch=3)
    seen_logits, env_actions = [], []
    fwd = policy.forward

    def rec(*a, **k):
        out = fwd(*a, **k)
        seen_logits.append(out.action_logits[:, -1].cpu().numpy().copy())
        return out
    policy.forward = rec
    rng = np.random.default_rng(3)

    class VecEnv:
        num_envs = 3
        action_space, observation_space = Box(-1, 1, (4,), np.float32), Box(-1, 1, (39,), np.float32)

        def reset(self):
            return rng.uniform(-1, 1, (3, 39)).astype(np.float32)

        def step(self, actions):
            env_actions.append(np.asarray(actions).reshape(3, -1).copy())
            done = np.full(3, len(env_actions) % 4 == 0)
            return self.reset(), np.ones(3, np.float32), done, [{} for _ in range(3)]

    kw = dict(temperature=1.0, top_k=0, top_p=0.5)
    agent = DiscreteDecisionXLSTM(policy, target_return=0.5, reward_scale=200.0, a_sample_kwargs=kw, a_sample_seed=8)
    custom_evaluate_policy(agent, VecEnv(), n_eval_episodes=3, warn=False)
    assert len(env_actions) == len(seen_logits) > 0
    for lg, act in zip(seen_logits, env_actions):
        cand = host_candidates(lg, 0.5, 0)                       # lg [3, act_dim, n]: one env per block
        k = act.shape[1]
        for b in range(3):
            assert all(cand[b, j, int(act[b, j])] for j in range(k)), (b, act[b])
    out = agent.predict_batch(policy, torch.from_numpy(rng.uniform(-1, 1, (3, 39)).astype(np.float32)),
                              torch.full((3,), 0.5), 4)
    assert out.dtype == torch.long and tuple(out.shape) == (3, cfg.act_dim)


@gpu
def test_disarmed_steps_equal_never_armed_steps():
    cfg, eng = _engine("toy128", 5)
    for flags in (0, L.XL_FLAG_GRAPH, L.XL_FLAG_DISCRETE | L.XL_FLAG_GRAPH):
        ref = _run_steps(eng, cfg, 5, 3, flags)
        eng.set_sampling(**KW)
        _run_steps(eng, cfg, 5, 1, flags)
        eng.set_sampling(None)
        got = _run_steps(eng, cfg, 5, 3, flags)
        for a, b in zip(ref, got):
            for k in a:
                assert torch.equal(a[k], b[k]), (flags, k)
    eng.close()
