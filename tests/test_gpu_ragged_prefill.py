"""Ragged context prefill (xl_prefill_ragged / xl_policy_prefill_ragged): a context length per env, envs without a
context left untouched. Checked against the oracle stepping each env over its own tokens, and against the library's
uniform prefill of each env alone. The argument checks run without a GPU."""
import numpy as np
import pytest
import torch

from lram_b200 import _lib as L
from lram_b200.config import preset
from lram_b200.synth import make_state_dict, make_stream

gpu = pytest.mark.gpu
REL_TOL = 1e-3


class NoLib:
    def __getattr__(self, name):
        raise AssertionError(f"{name} reached the library")


class _State:
    def __init__(self, B):
        self.B = B


# ---- CPU: argument checks -------------------------------------------------------------------------------------------
_BAD_LENGTHS = [[3, 2], [3, 2, 1, 0], [3, -1, 2], [3, 9, 2], [1.5, 2, 3], np.array([1.0, 2.0, 3.0]),
                torch.tensor([1.0, 2.0, 3.0]), [True, False, True], np.array([[1, 2, 3]]), ["a", "b", "c"]]


def _nolib_engine():
    from lram_b200.engine import XLSTMEngine
    eng = XLSTMEngine.__new__(XLSTMEngine)
    eng.cfg, eng.lib, eng.handle = preset("toy128"), NoLib(), None
    return eng


def test_prefill_lengths_rejected_before_the_library():
    eng = _nolib_engine()
    cfg, B, S = eng.cfg, 3, 8
    x = torch.zeros(B, S, cfg.d)
    states, rtg = torch.zeros(B, S, cfg.state_dim), torch.zeros(B, S)
    for bad in _BAD_LENGTHS:
        with pytest.raises(ValueError):
            eng.prefill(_State(B), x, lengths=bad)
        with pytest.raises(ValueError):
            eng.policy_prefill(_State(B), states, rtg, lengths=bad)


def test_check_lengths_accepts_sequences_arrays_and_cpu_int_tensors():
    from lram_b200.engine import check_lengths
    for ok in ([3, 0, 8], np.array([3, 0, 8], np.int64), torch.tensor([3, 0, 8], dtype=torch.int32), (3, 0, 8)):
        got = check_lengths(ok, 3, 8)
        assert got.dtype == np.int32 and got.flags["C_CONTIGUOUS"] and got.tolist() == [3, 0, 8]


def test_prefill_context_lengths_rejected_before_the_library():
    from lram_b200.rollout import BatchedRollout
    eng = _nolib_engine()
    ro = BatchedRollout.__new__(BatchedRollout)
    ro.engine, ro.B, ro.state = eng, 3, _State(3)
    states, rtg = np.zeros((3, 8, eng.cfg.state_dim), np.float32), np.zeros((3, 8), np.float32)
    for bad in _BAD_LENGTHS:
        with pytest.raises(ValueError):
            ro.prefill_context(states, rtg, lengths=bad)


# ---- GPU helpers ----------------------------------------------------------------------------------------------------
def _engine(name, B, seed=0, **over):
    from lram_b200.engine import XLSTMEngine
    cfg = preset(name, **over)
    sd = make_state_dict(cfg, seed=seed)
    return cfg, sd, XLSTMEngine(cfg, sd, max_batch=B)


def _rel(a, b):
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _env_pkv(pkv, b):
    """One env of a past_key_values dict (sLSTM planes are [4, B, d])."""
    out = {}
    for blk, st in pkv.items():
        out[blk] = {}
        for k, v in st.items():
            if k == "slstm_state":
                out[blk][k] = v[:, b:b + 1].clone()
            else:
                out[blk][k] = tuple(t[b:b + 1].clone() for t in v)
    return out


def _slots(cfg, cache, b):
    """Raw bytes of env b's state slot, part by part."""
    out = []
    for i in range(cfg.num_blocks):
        if cfg.is_slstm(i):
            out += [cache.view(i, L.XL_STATE_SLSTM)[:, b].clone(), cache.view(i, L.XL_STATE_CONV)[b].clone()]
        else:
            out += [cache.view(i, p)[b].clone() for p in (L.XL_STATE_C, L.XL_STATE_N, L.XL_STATE_M, L.XL_STATE_CONV)]
    return out


def _slots_equal(a, b):
    return all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(a, b))


def _copy(eng, cache):
    c = eng.new_state(cache.B)
    c.buf.copy_(cache.buf)
    return c


def _assert_env_matches_oracle(cfg, exp, ora, tol=REL_TOL):
    """exp / ora: one env's past_key_values (library export / oracle)."""
    for i in range(cfg.num_blocks):
        eo, oo = exp[f"block_{i}"], ora[f"block_{i}"]
        assert _rel(eo["conv_state"][0].cpu(), oo["conv_state"][0]) < 1e-5, f"block {i} conv"
        if cfg.is_slstm(i):
            se, so = eo["slstm_state"].cpu(), oo["slstm_state"]
            for part, nm in enumerate("ycnm"):
                assert _rel(se[part], so[part]) < tol, f"block {i} sLSTM {nm}"
            continue
        c, n, m = oo["mlstm_state"]
        ce, ne, me = eo["mlstm_state"]
        assert _rel(ce.cpu(), c) < tol and _rel(ne.cpu(), n) < tol, f"block {i}"
        assert (me.cpu() - m).abs().max() < 1e-4, f"block {i} m"


def _assert_env_states_close(cfg, a, b, tol=1e-4):
    for i in range(cfg.num_blocks):
        ea, eb = a[f"block_{i}"], b[f"block_{i}"]
        parts = [ea["slstm_state"]] if cfg.is_slstm(i) else list(ea["mlstm_state"])
        refs = [eb["slstm_state"]] if cfg.is_slstm(i) else list(eb["mlstm_state"])
        for x, y in zip(parts + [ea["conv_state"][0]], refs + [eb["conv_state"][0]]):
            x, y = x.cpu(), y.cpu()
            assert _rel(x, y) < tol or (x - y).abs().max() < 1e-5, f"block {i}"


def _oracle_ragged(cfg, sd, x0, x, lengths):
    """Oracle: 2 warm-up tokens for every env, then each env stepped over its own lengths[b] tokens. -> hidden rows
    [B, S, d] (rows past an env's length are 0) and one past_key_values per env."""
    from oracle import xlstm_oracle as O
    ora = O.OracleEncoder(cfg, sd)
    B, S = x.shape[:2]
    _, pkv = ora.forward_cached(x0, None)
    hid = torch.zeros(B, S, cfg.d)
    envs = [_env_pkv(pkv, b) if lengths[b] == 0 else None for b in range(B)]
    for t in range(max(lengths)):
        r, pkv = ora.forward_cached(x[:, t:t + 1], pkv)
        for b in range(B):
            if t < lengths[b]:
                hid[b, t] = r[b, 0]
            if t + 1 == lengths[b]:
                envs[b] = _env_pkv(pkv, b)
    return hid, envs


def _warm(eng, cfg, B, g):
    """A cache after two step tokens (a non-zero state) and those tokens."""
    x0 = torch.randn(B, 2, cfg.d, generator=g)
    cache = eng.new_state(B)
    eng.encoder_step(cache, x0.cuda())
    return cache, x0


# ---- 1 + 3: every cell against the oracle; pads never read ----------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["16M", "toy128"])
def test_ragged_prefill_every_cell_vs_oracle(name):
    B, S, lengths = 5, 304, [304, 0, 129, 3, 128]
    cfg, sd, eng = _engine(name, B)
    g = torch.Generator().manual_seed(3)
    warm, x0 = _warm(eng, cfg, B, g)
    x = torch.randn(B, S, cfg.d, generator=g)
    hid_o, env_o = _oracle_ragged(cfg, sd, x0, x, lengths)
    slot1 = _slots(cfg, warm, 1)
    xz, xn = x.clone(), x.clone()
    for b, n in enumerate(lengths):
        xz[b, n:] = 0.0
        xn[b, n:] = float("nan")
        xn[b, n::2] = float("inf")
    launches = {}
    for cell in (2, 1, 0):
        eng.set_option("prefill_cell", cell)
        cache = _copy(eng, warm)
        eng.launch_count()
        hs = eng.prefill(cache, xn.cuda(), lengths=lengths)
        torch.cuda.synchronize()
        launches[cell] = eng.launch_count()
        hs = hs.cpu()
        for b, n in enumerate(lengths):
            assert torch.all(hs[b, n:] == 0), (cell, b)
            if n:
                assert _rel(hs[b, :n], hid_o[b, :n]) < REL_TOL, (cell, b)
        exp = cache.to_past_key_values()
        for b, n in enumerate(lengths):
            _assert_env_matches_oracle(cfg, _env_pkv(exp, b), env_o[b])
        assert _slots_equal(_slots(cfg, cache, 1), slot1), cell
        # pads hold NaN / inf above: zeros there give bit-identical results
        cz = _copy(eng, warm)
        hz = eng.prefill(cz, xz.cuda(), lengths=lengths)
        torch.cuda.synchronize()
        assert torch.equal(hz.cpu(), hs) and torch.equal(cz.buf, cache.buf), cell
    eng.set_option("prefill_cell", 2)
    if name == "16M":
        assert launches[2] > launches[1]        # the tcgen05 cell ran
    eng.close()


# ---- 2: outer chunks and the shrinking prefix -----------------------------------------------------------------------
def _uniform_alone(eng, wpkv, x, b, n):
    """Env b of the starting state `wpkv` prefilled alone (B = 1, the uniform call) over its first n tokens -> its
    past_key_values."""
    one = eng.new_state(1)
    one.load_past_key_values(_env_pkv(wpkv, b))
    if n:
        eng.prefill(one, x[b:b + 1, :n].contiguous().cuda(), want_hidden=False)
    torch.cuda.synchronize()
    return one.to_past_key_values()


@gpu
@pytest.mark.parametrize("rows,lengths", [(384, [400, 96, 250, 37]), (16384, [5000, 3000])])
def test_ragged_prefill_outer_chunks_match_single_env_prefills(rows, lengths):
    """prefill_rows = 384: chunks of 96 tokens at 4 envs, 192 at 2, 384 at 1; the env of 96 ends exactly on the first
    outer-chunk boundary, the others inside chunks. Default rows at 2 envs: 8192-token chunks, the env of 3000 ends inside
    the second 2048-token super-chunk of the gate scan."""
    B = len(lengths)
    cfg, sd, eng = _engine("16M", B)
    g = torch.Generator().manual_seed(7)
    warm, _ = _warm(eng, cfg, B, g)
    x = torch.randn(B, max(lengths), cfg.d, generator=g)
    eng.set_option("prefill_rows", rows)
    cache = _copy(eng, warm)
    eng.prefill(cache, x.cuda(), want_hidden=False, lengths=lengths)
    torch.cuda.synchronize()
    exp, wpkv = cache.to_past_key_values(), warm.to_past_key_values()
    for b, n in enumerate(lengths):
        _assert_env_states_close(cfg, _env_pkv(exp, b), _uniform_alone(eng, wpkv, x, b, n))
    eng.close()


# ---- 4: order does not matter ---------------------------------------------------------------------------------------
@gpu
def test_ragged_prefill_env_order_is_irrelevant():
    B, S, lengths = 6, 200, [200, 17, 0, 130, 64, 130]
    cfg, sd, eng = _engine("16M", B)
    g = torch.Generator().manual_seed(9)
    warm, _ = _warm(eng, cfg, B, g)
    x = torch.randn(B, S, cfg.d, generator=g)
    perm = [3, 5, 0, 2, 4, 1]
    ca = _copy(eng, warm)
    ha = eng.prefill(ca, x.cuda(), lengths=lengths)
    wb = eng.new_state(B)                                # env k of the shuffled batch = env perm[k] of the first
    pkv = warm.to_past_key_values()
    shuffled = {blk: {k: (v[:, perm] if k == "slstm_state" else tuple(t[perm] for t in v)) for k, v in st.items()}
                for blk, st in pkv.items()}
    wb.load_past_key_values(shuffled)
    hb = eng.prefill(wb, x[perm].cuda(), lengths=[lengths[b] for b in perm])
    torch.cuda.synchronize()
    for k, b in enumerate(perm):
        assert torch.equal(hb[k].cpu(), ha[b].cpu()), (k, b)
        assert _slots_equal(_slots(cfg, wb, k), _slots(cfg, ca, b)), (k, b)
    eng.close()


# ---- 5: uniform lengths are the uniform call -------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("S", [37, 304])
def test_ragged_prefill_uniform_lengths_equal_uniform_call(S):
    B = 3
    cfg, sd, eng = _engine("16M", B)
    g = torch.Generator().manual_seed(13)
    warm, _ = _warm(eng, cfg, B, g)
    x = torch.randn(B, S, cfg.d, generator=g).cuda()
    ca, cb = _copy(eng, warm), _copy(eng, warm)
    ha = eng.prefill(ca, x)
    hb = eng.prefill(cb, x, lengths=[S] * B)
    torch.cuda.synchronize()
    assert torch.equal(ha, hb) and torch.equal(ca.buf, cb.buf)
    Tn = S // 3 + 1
    states, rtg, _ = make_stream(cfg, range(B), Tn, domains="mixed", seed=4)
    st = torch.from_numpy(np.ascontiguousarray(states.transpose(1, 0, 2))).cuda()
    rt = torch.from_numpy(np.ascontiguousarray(rtg.T)).cuda()
    pa, pb = eng.new_state(B), eng.new_state(B)
    eng.policy_prefill(pa, st, rt)
    eng.policy_prefill(pb, st, rt, lengths=np.full(B, Tn))
    torch.cuda.synchronize()
    assert torch.equal(pa.buf, pb.buf)
    eng.close()


# ---- 6: policy form ---------------------------------------------------------------------------------------------------
@gpu
def test_policy_prefill_ragged_equals_per_env_stepping():
    B, Tn, Tr, lengths = 4, 100, 4, [100, 0, 23, 57]
    cfg, sd, eng = _engine("16M", B)
    states, rtg, _ = make_stream(cfg, range(B), Tn + Tr, domains="mixed", seed=21)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    ctx_s = states[:Tn].transpose(1, 0, 2).copy()          # [B, Tn, sd]
    ctx_r = rtg[:Tn].T.copy()
    for b, n in enumerate(lengths):                       # pads are never read
        ctx_s[b, n:] = np.nan
        ctx_r[b, n:] = np.inf
    pre = eng.new_state(B)
    eng.policy_prefill(pre, dev(ctx_s), dev(ctx_r), lengths=lengths)
    singles = []
    for b, n in enumerate(lengths):
        one = eng.new_state(1)
        for t in range(n):
            eng.policy_step(one, dev(states[t, b:b + 1]), dev(rtg[t, b:b + 1]))
        singles.append(one)
    torch.cuda.synchronize()
    exp = pre.to_past_key_values()
    for b in range(B):
        _assert_env_states_close(cfg, _env_pkv(exp, b), singles[b].to_past_key_values())
    # each env then steps on from its own context: same action tokens as the single-env caches
    for t in range(Tr):
        s_t = np.stack([states[lengths[b] + t, b] for b in range(B)])
        r_t = np.array([rtg[lengths[b] + t, b] for b in range(B)], np.float32)
        out = eng.policy_step(pre, dev(s_t), dev(r_t))
        for b in range(B):
            o1 = eng.policy_step(singles[b], dev(s_t[b:b + 1]), dev(r_t[b:b + 1]))
            torch.cuda.synchronize()
            assert torch.equal(out["action_tokens"][b].cpu(), o1["action_tokens"][0].cpu()), (t, b)
    eng.close()


@gpu
def test_policy_prefill_ragged_leaves_sampler_step_and_token_ring_alone():
    B, Tn, lengths = 4, 40, [40, 0, 9, 31]
    cfg, sd, eng = _engine("16M", B)
    states, rtg, _ = make_stream(cfg, range(B), Tn + 1, domains="mixed", seed=5)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    ring = torch.full((6, B, cfg.act_dim), -1, dtype=torch.int32, device="cuda")
    eng.set_token_ring(ring, next_slot=2)
    kw = dict(temperature=1.0, top_k=0, top_p=0.5, seed=1234)
    eng.set_sampling(**kw, step0=17)
    cache = eng.new_state(B)
    eng.policy_prefill(cache, dev(states[:Tn].transpose(1, 0, 2)), dev(rtg[:Tn].T), lengths=lengths)
    out = eng.policy_step(cache, dev(states[Tn]), dev(rtg[Tn]), want_logits=True)
    torch.cuda.synchronize()
    tok, _ = eng.sample_actions(out["action_logits"], step=17, **kw)
    assert torch.equal(out["action_tokens"], tok)
    assert torch.equal(ring[2], out["action_tokens"])
    assert bool((ring[[0, 1, 3, 4, 5]] == -1).all())
    eng.set_sampling(None)
    eng.set_token_ring(None)
    eng.close()


# ---- 7: sLSTM stacks --------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name,lengths", [("toy128-ms", [30, 0, 2, 17, 3]), ("48M-ms", [40, 3, 0])])
def test_ragged_prefill_slstm_stacks_vs_oracle(name, lengths):
    B, S = len(lengths), max(lengths)
    cfg, sd, eng = _engine(name, B)
    g = torch.Generator().manual_seed(17)
    warm, x0 = _warm(eng, cfg, B, g)
    x = torch.randn(B, S, cfg.d, generator=g)
    hid_o, env_o = _oracle_ragged(cfg, sd, x0, x, lengths)
    zero = [b for b, n in enumerate(lengths) if n == 0][0]
    slot0 = _slots(cfg, warm, zero)
    cache = _copy(eng, warm)
    hs = eng.prefill(cache, x.cuda(), lengths=lengths).cpu()
    torch.cuda.synchronize()
    exp = cache.to_past_key_values()
    for b, n in enumerate(lengths):
        assert torch.all(hs[b, n:] == 0)
        if n:
            assert _rel(hs[b, :n], hid_o[b, :n]) < REL_TOL, b
        _assert_env_matches_oracle(cfg, _env_pkv(exp, b), env_o[b])
    assert _slots_equal(_slots(cfg, cache, zero), slot0)
    eng.close()


# ---- 8: rollout -------------------------------------------------------------------------------------------------------
@gpu
def test_batched_rollout_ragged_context_and_subset_reprime():
    from lram_b200.rollout import BatchedRollout
    from lram_b200.synth import SyntheticEnvBatch
    B, Tn, Tr, lengths = 4, 30, 5, [30, 0, 11, 26]
    cfg, sd, eng = _engine("16M", B, seed=8)
    ctx_s, ctx_r, _ = make_stream(cfg, range(B), Tn, domains="mixed", seed=55)
    res = {}
    for tag in ("ragged", "stepped"):
        envs = SyntheticEnvBatch(cfg, range(B), domains="mixed", ep_len=50, seed=77)
        ro = BatchedRollout(eng, envs, use_graph=True)
        if tag == "ragged":
            ro.prefill_context(ctx_s.transpose(1, 0, 2), ctx_r.T, lengths=lengths)
        else:
            eng.reset(ro.state)
            for b, n in enumerate(lengths):
                one = eng.new_state(1)
                for t in range(n):
                    eng.policy_step(one, torch.from_numpy(ctx_s[t, b:b + 1]).cuda(),
                                    torch.from_numpy(ctx_r[t, b:b + 1]).cuda())
                torch.cuda.synchronize()
                pkv = ro.state.to_past_key_values()
                mine = one.to_past_key_values()
                for blk in pkv:
                    for k, v in pkv[blk].items():
                        for full, part in zip(v if isinstance(v, tuple) else (v,),
                                              mine[blk][k] if isinstance(v, tuple) else (mine[blk][k],)):
                            full[b:b + 1] = part
                ro.state.load_past_key_values(pkv)
        res[tag] = ro.run(Tr, record=True, keep_state=True)
        res[tag + "_ro"] = ro
    assert np.array_equal(res["ragged"]["tokens"], res["stepped"]["tokens"])
    assert np.array_equal(res["ragged"]["actions"], res["stepped"]["actions"])
    # re-prime envs 1 and 2 of the running batch: envs 0 and 3 keep every byte
    ro = res["ragged_ro"]
    before = [_slots(cfg, ro.state, b) for b in range(B)]
    ro.prefill_context(ctx_s.transpose(1, 0, 2), ctx_r.T, lengths=[0, 7, 12, 0])
    torch.cuda.synchronize()
    for b in (0, 3):
        assert _slots_equal(_slots(cfg, ro.state, b), before[b]), b
    assert not _slots_equal(_slots(cfg, ro.state, 1), before[1])
    eng.close()


# ---- 9: large batch ---------------------------------------------------------------------------------------------------
@gpu
def test_ragged_prefill_large_batch_vs_single_env_prefills():
    B, S = 128, 160
    rng = np.random.default_rng(2024)
    lengths = rng.integers(0, S + 1, B)
    lengths[:3] = [S, 0, 1]
    cfg, sd, eng = _engine("48M", B)
    g = torch.Generator().manual_seed(19)
    warm, _ = _warm(eng, cfg, B, g)
    x = torch.randn(B, S, cfg.d, generator=g)
    cache = _copy(eng, warm)
    eng.prefill(cache, x.cuda(), want_hidden=False, lengths=lengths)
    torch.cuda.synchronize()
    exp, wpkv = cache.to_past_key_values(), warm.to_past_key_values()
    for b in [0, 1, 2] + rng.choice(np.arange(3, B), 5, replace=False).tolist():
        _assert_env_states_close(cfg, _env_pkv(exp, b), _uniform_alone(eng, wpkv, x, b, int(lengths[b])))
    eng.close()


# ---- 10: shapes outside the sequence path --------------------------------------------------------------------------
@gpu
def test_ragged_prefill_outside_sequence_path_is_rejected_untouched():
    # the step path has KS = 3 kernels for 1 and 3 tokens per call: warm one token at a time, S = 3 for the uniform call
    B, S = 3, 3
    cfg, sd, eng = _engine("toy128", B, conv1d_kernel_size=3)
    g = torch.Generator().manual_seed(29)
    warm = eng.new_state(B)
    for _ in range(2):
        eng.encoder_step(warm, torch.randn(B, 1, cfg.d, generator=g).cuda())
    x = torch.randn(B, S, cfg.d, generator=g).cuda()
    cache = _copy(eng, warm)
    with pytest.raises(L.XLError) as ei:
        eng.prefill(cache, x, lengths=[3, 0, 2])
    assert ei.value.code == L.XL_ERR_UNSUPPORTED
    torch.cuda.synchronize()
    assert torch.equal(cache.buf, warm.buf)
    ref = _copy(eng, warm)
    ha = eng.prefill(ref, x)
    hb = eng.prefill(cache, x, lengths=[S] * B)
    torch.cuda.synchronize()
    assert torch.equal(ha, hb) and torch.equal(ref.buf, cache.buf)
    eng.close()
