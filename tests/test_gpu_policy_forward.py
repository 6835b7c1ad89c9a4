"""Sequence forward of the policy (xl_policy_forward / XLSTMEngine.policy_forward / the model's non-cache forward): the
action outputs of every timestep of whole trajectories in one chunkwise pass. Checked against the oracle stepping each
env, against the library's own prefill and policy steps, and at the Python layer. The argument checks run without a GPU.

Near-ties: the chunkwise prefill and recurrent steps agree to rounding, so a token may flip only where the reference's
top-two logits of that row are closer than TIE; every such flip is counted and printed."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from lram_b200 import _lib as L
from lram_b200.config import preset
from lram_b200.synth import make_state_dict, make_stream

gpu = pytest.mark.gpu
REL_TOL = 1e-3
TIE = 1e-4


class NoLib:
    def __getattr__(self, name):
        raise AssertionError(f"{name} reached the library")


class _State:
    def __init__(self, B):
        self.B = B


def _nolib_engine(device="cuda:0"):
    from lram_b200.engine import XLSTMEngine
    eng = XLSTMEngine.__new__(XLSTMEngine)
    eng.cfg, eng.lib, eng.handle, eng.device = preset("toy128"), NoLib(), None, torch.device(device)
    return eng


# ---- CPU: argument checks -------------------------------------------------------------------------------------------
def test_policy_forward_arguments_rejected_before_the_library():
    eng = _nolib_engine()
    cfg, B, Tn = eng.cfg, 3, 8
    states, rtg = torch.zeros(B, Tn, cfg.state_dim), torch.zeros(B, Tn)
    for bad in ([3, 2], [3, -1, 2], [3, 9, 2], [1.5, 2, 3], torch.tensor([1.0, 2.0, 3.0]), [True, False, True]):
        with pytest.raises(ValueError):
            eng.policy_forward(_State(B), states, rtg, lengths=bad)
    ok = torch.zeros(B, Tn, cfg.act_dim, dtype=torch.int32)
    for bad in (ok.float(), ok.bool(), ok[:, :, :2], ok[:2], ok.numpy(), ok):   # the last one: on the host, not cuda:0
        with pytest.raises(ValueError):
            eng.policy_forward(_State(B), states, rtg, targets=bad)
    eng = _nolib_engine("cpu")                       # targets on the engine's device: only the range is wrong
    for v in (-2, cfg.num_actions, 10 ** 6):
        bad = ok.clone().long()
        bad[1, 2, 3] = v
        with pytest.raises(ValueError):
            eng.policy_forward(_State(B), states, rtg, targets=bad)


def test_image_states_and_grad_inputs_raise_not_implemented():
    from lram_b200 import decision_xlstm as DX
    cfg = preset("toy128")
    model = DX.MultiDomainDiscreteDecisionXLSTMModel(cfg)
    B, T = 2, 3
    frames = torch.zeros(B, T, 3, 64, 64)
    with pytest.raises(NotImplementedError):
        model(states=frames, actions=torch.zeros(B, T, 1), returns_to_go=torch.zeros(B, T, 1),
              use_inference_cache=False)
    enc = DX.FusedXLSTMEncoder(config=cfg)
    x = torch.zeros(B, 6, cfg.d, requires_grad=True)
    with pytest.raises(NotImplementedError):
        enc(inputs_embeds=x, use_cache=False)


# ---- GPU helpers ----------------------------------------------------------------------------------------------------
def _engine(name, B, seed=0, **over):
    from lram_b200.engine import XLSTMEngine
    cfg = preset(name, **over)
    sd = make_state_dict(cfg, seed=seed)
    return cfg, sd, XLSTMEngine(cfg, sd, max_batch=B)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _inputs(cfg, B, Tn, seed):
    """states [B, Tn, sd], rtg [B, Tn], rewards [B, Tn] (numpy fp32)."""
    s, r, _ = make_stream(cfg, range(B), Tn, domains="mixed", seed=seed)
    rew = np.random.default_rng(seed).normal(0.0, 0.5, (B, Tn)).astype(np.float32)
    return s.transpose(1, 0, 2).copy(), r.T.copy(), rew


def _warm(eng, cfg, B, seed):
    """A non-zero start state: three policy steps from zero."""
    s, r, w = _inputs(cfg, B, 3, seed + 1000)
    cache = eng.new_state(B)
    for t in range(3):
        eng.policy_step(cache, _dev(s[:, t]), _dev(r[:, t]), _dev(w[:, t]))
    torch.cuda.synchronize()
    return cache


def _copy(eng, cache):
    c = eng.new_state(cache.B)
    c.buf.copy_(cache.buf)
    return c


def _cpu(pkv):
    return {blk: {k: (v.cpu() if torch.is_tensor(v) else tuple(t.cpu() for t in v)) for k, v in st.items()}
            for blk, st in pkv.items()}


def _env_pkv(pkv, b):
    return {blk: {k: (v[:, b:b + 1].clone() if k == "slstm_state" else tuple(t[b:b + 1].clone() for t in v))
                  for k, v in st.items()} for blk, st in pkv.items()}


def _rel(a, b):
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _slots(cfg, cache, b):
    out = []
    for i in range(cfg.num_blocks):
        if cfg.is_slstm(i):
            out += [cache.view(i, L.XL_STATE_SLSTM)[:, b].clone(), cache.view(i, L.XL_STATE_CONV)[b].clone()]
        else:
            out += [cache.view(i, p)[b].clone() for p in (L.XL_STATE_C, L.XL_STATE_N, L.XL_STATE_M, L.XL_STATE_CONV)]
    return out


def _slots_equal(a, b):
    return all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(a, b))


_ORACLE = {}


def _oracle(name, cfg, sd, pkv0, s, r, w):
    """OraclePolicy.step over every timestep from pkv0 -> full head logits [B, Tn, act_dim, num_actions] and the final
    past_key_values. Cached per case: continuous and discrete read the same logits."""
    from oracle.xlstm_oracle import OraclePolicy
    key = (name, s.shape)
    if key not in _ORACLE:
        ora = OraclePolicy(cfg, sd)
        pkv, lg = pkv0, []
        for t in range(s.shape[1]):
            o = ora.step(torch.from_numpy(s[:, t]), torch.from_numpy(r[:, t]), torch.from_numpy(w[:, t]),
                         past_key_values=pkv)
            pkv = o["past_key_values"]
            lg.append(o["action_logits"])
        _ORACLE.clear()
        _ORACLE[key] = (torch.stack(lg, 1), pkv)
    return _ORACLE[key]


def _argmax_rows(cfg, logits, discrete):
    """Rows the argmax reads: [..., act_dim, num_actions] -> discrete [..., 1, discrete_actions]."""
    return logits[..., :1, :cfg.discrete_actions] if discrete else logits


def _check_tokens(cfg, tok, ref_logits, discrete, what):
    """tok [..., act_dim] from the library; ref_logits [..., act_dim, num_actions]. Flips only at near-ties."""
    rows = _argmax_rows(cfg, ref_logits.double(), discrete)
    ref = rows.argmax(-1)
    top2 = rows.topk(2, dim=-1).values
    margin = top2[..., 0] - top2[..., 1]
    got = tok[..., :1] if discrete else tok
    flips = got.long().cpu() != ref.cpu()
    n = int(flips.sum())
    if n:
        print(f"{what}: {n} near-tie token flip(s) of {flips.numel()}")
    assert bool((margin.cpu()[flips] < TIE).all()), f"{what}: token differs away from a near-tie"
    return n


def _assert_state_close(cfg, exp, ora, tol=REL_TOL):
    for i in range(cfg.num_blocks):
        eo, oo = exp[f"block_{i}"], ora[f"block_{i}"]
        assert _rel(eo["conv_state"][0].cpu(), oo["conv_state"][0]) < 1e-5, f"block {i} conv"
        if cfg.is_slstm(i):
            for part in range(4):
                assert _rel(eo["slstm_state"][part].cpu(), oo["slstm_state"][part]) < tol, f"block {i} sLSTM"
            continue
        (c, n, m), (ce, ne, me) = oo["mlstm_state"], eo["mlstm_state"]
        assert _rel(ce.cpu(), c) < tol and _rel(ne.cpu(), n) < tol, f"block {i}"
        assert (me.cpu() - m).abs().max() < 1e-4, f"block {i} m"


def _shape_logits(cfg, lg, discrete):
    B, Tn = lg.shape[:2]
    return lg.view(B, Tn, 1, cfg.num_actions) if discrete else lg.view(B, Tn, cfg.act_dim, cfg.num_actions)


# ---- 1 + 2: against the oracle, state bytes equal to the prefill ----------------------------------------------------
_CASES = [("16M", (2, 1, 0)), ("toy128", (2, 1, 0)), ("toy128-ms", (2,)), ("48M-ms", (2,))]


@gpu
@pytest.mark.parametrize("name,cells", _CASES)
@pytest.mark.parametrize("Tn", [45, 200])
def test_policy_forward_vs_oracle_every_cell(name, cells, Tn):
    B = 2
    cfg, sd, eng = _engine(name, B, seed=3)
    warm = _warm(eng, cfg, B, seed=5)
    s, r, w = _inputs(cfg, B, Tn, seed=11)
    ref_lg, ref_pkv = _oracle(name, cfg, sd, _cpu(warm.to_past_key_values()), s, r, w)
    flips = 0
    for cell in cells:
        eng.set_option("prefill_cell", cell)
        pre = _copy(eng, warm)
        eng.policy_prefill(pre, _dev(s), _dev(r), _dev(w))
        for discrete in (False, True):
            cache = _copy(eng, warm)
            out = eng.policy_forward(cache, _dev(s), _dev(r), _dev(w), discrete=discrete, want_logits=True)
            torch.cuda.synchronize()
            assert torch.equal(cache.buf, pre.buf), (cell, discrete)           # bit-identical to xl_policy_prefill
            lg = _shape_logits(cfg, out["action_logits"].cpu(), discrete)
            ref = ref_lg[:, :, :1] if discrete else ref_lg
            assert _rel(lg, ref) < REL_TOL, (cell, discrete)
            flips += _check_tokens(cfg, out["action_tokens"], ref, discrete, f"{name} cell {cell} d={discrete}")
            if discrete:
                assert bool((out["action_tokens"][..., 1:] == -1).all() and (out["action_preds"][..., 1:] == 0).all())
                assert torch.equal(out["action_preds"][..., 0], out["action_tokens"][..., 0].float())
        _assert_state_close(cfg, pre.to_past_key_values(), ref_pkv)
    eng.set_option("prefill_cell", 2)
    print(f"{name} Tn={Tn}: {flips} near-tie flips")
    eng.close()


# ---- 3: all tail ----------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("discrete", [False, True])
def test_policy_forward_short_equals_eager_steps(discrete):
    B, Tn = 3, 5
    cfg, sd, eng = _engine("16M", B, seed=4)
    warm = _warm(eng, cfg, B, seed=6)
    s, r, w = _inputs(cfg, B, Tn, seed=12)
    cache = _copy(eng, warm)
    out = eng.policy_forward(cache, _dev(s), _dev(r), _dev(w), discrete=discrete, want_logits=True)
    step = _copy(eng, warm)
    flags = L.XL_FLAG_DISCRETE if discrete else 0
    for t in range(Tn):
        o = eng.policy_step(step, _dev(s[:, t]), _dev(r[:, t]), _dev(w[:, t]), flags=flags, want_logits=True)
        torch.cuda.synchronize()
        cols = slice(0, 1) if discrete else slice(None)
        assert torch.equal(out["action_tokens"][:, t, cols], o["action_tokens"][:, cols]), t
        assert torch.equal(out["action_preds"][:, t, cols], o["action_preds"][:, cols]), t
        assert torch.equal(out["action_logits"][:, t], o["action_logits"]), t
    assert torch.equal(cache.buf, step.buf)
    eng.close()


# ---- 4: ragged lengths ----------------------------------------------------------------------------------------------
@gpu
def test_policy_forward_ragged():
    B, Tn, lengths = 6, 200, [200, 0, 45, 7, 133, 45]
    cfg, sd, eng = _engine("16M", B, seed=7)
    warm = _warm(eng, cfg, B, seed=8)
    s, r, w = _inputs(cfg, B, Tn, seed=13)
    sn, rn, wn = s.copy(), r.copy(), w.copy()
    for b, n in enumerate(lengths):                     # never read
        sn[b, n:], rn[b, n:], wn[b, n:] = np.nan, np.nan, np.nan
    tg = torch.randint(-1, cfg.num_actions, (B, Tn, cfg.act_dim), generator=torch.Generator().manual_seed(1)).cuda()
    cache = _copy(eng, warm)
    out = eng.policy_forward(cache, _dev(sn), _dev(rn), _dev(wn), lengths=lengths, targets=tg, want_logits=True)
    pre = _copy(eng, warm)
    eng.policy_prefill(pre, _dev(sn), _dev(rn), _dev(wn), lengths=lengths)
    torch.cuda.synchronize()
    assert torch.equal(cache.buf, pre.buf)                                     # == xl_policy_prefill_ragged
    assert _slots_equal(_slots(cfg, cache, 1), _slots(cfg, warm, 1))
    for b, n in enumerate(lengths):
        assert bool((out["action_tokens"][b, n:] == -1).all()), b
        for k in ("action_preds", "action_logits", "action_logprobs"):
            assert bool((out[k][b, n:] == 0).all()), (b, k)
    # each env against its own uniform forward (B = 1)
    wpkv = warm.to_past_key_values()
    for b, n in enumerate(lengths):
        if not n:
            continue
        one = eng.new_state(1)
        one.load_past_key_values(_env_pkv(wpkv, b))
        o1 = eng.policy_forward(one, _dev(s[b:b + 1, :n]), _dev(r[b:b + 1, :n]), _dev(w[b:b + 1, :n]),
                                targets=tg[b:b + 1, :n].contiguous(), want_logits=True)
        torch.cuda.synchronize()
        lg1 = _shape_logits(cfg, o1["action_logits"].cpu(), False)
        assert _rel(out["action_logits"][b, :n].cpu(), o1["action_logits"][0].cpu()) < REL_TOL, b
        _check_tokens(cfg, out["action_tokens"][b:b + 1, :n], lg1, False, f"ragged env {b}")
    # shuffled env order: bit-identical per env; envs 2 and 5 tie in length and swap places in the sorted plan
    perm = [3, 5, 0, 4, 1, 2]
    shuffled = {blk: {k: (v[:, perm] if k == "slstm_state" else tuple(t[perm] for t in v)) for k, v in st.items()}
                for blk, st in wpkv.items()}
    cs = eng.new_state(B)
    cs.load_past_key_values(shuffled)
    os_ = eng.policy_forward(cs, _dev(sn[perm]), _dev(rn[perm]), _dev(wn[perm]), lengths=[lengths[b] for b in perm],
                             targets=tg[perm].contiguous(), want_logits=True)
    torch.cuda.synchronize()
    for k, b in enumerate(perm):
        for key in out:
            assert torch.equal(os_[key][k], out[key][b]), (k, b, key)
        assert _slots_equal(_slots(cfg, cs, k), _slots(cfg, cache, b)), (k, b)
    eng.close()


# ---- 5: log-probabilities -------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("discrete", [False, True])
def test_policy_forward_logprobs(discrete):
    B, Tn = 3, 61
    cfg, sd, eng = _engine("16M", B, seed=9)
    s, r, w = _inputs(cfg, B, Tn, seed=14)
    tg = torch.randint(0, cfg.num_actions, (B, Tn, cfg.act_dim), generator=torch.Generator().manual_seed(2))
    tg[0, :, 5:] = -1
    tg[1, 3, 0] = -1
    tg = tg.cuda()
    out = eng.policy_forward(eng.new_state(B), _dev(s), _dev(r), _dev(w), discrete=discrete, targets=tg,
                             want_logits=True)
    torch.cuda.synchronize()
    lg = _shape_logits(cfg, out["action_logits"].cpu(), discrete).double()
    ls = torch.log_softmax(lg, dim=-1)
    t = tg.cpu().long()
    cols = 1 if discrete else cfg.act_dim
    exp = ls.gather(-1, t[..., :cols].clamp(min=0).unsqueeze(-1)).squeeze(-1)
    exp = torch.where(t[..., :cols] < 0, torch.zeros_like(exp), exp)
    got = out["action_logprobs"].cpu().double()
    assert (got[..., :cols] - exp).abs().max().item() < 1e-5
    assert bool((got[..., :cols][t[..., :cols] < 0] == 0).all())
    if discrete:
        assert bool((got[..., 1:] == 0).all())
    # a target == num_actions through the raw C call gives NaN; the Python layer would have refused it
    tg2 = tg.clone().to(torch.int32)
    tg2[2, 7, 0] = cfg.num_actions
    lp = torch.empty(B, Tn, cfg.act_dim, device="cuda")
    so = C.byref(L.XLSeqOutputs(tokens=None, actions=None, logits=None, targets=tg2.data_ptr(), logprobs=lp.data_ptr()))
    st = eng.new_state(B)
    sd_, rd, wd = _dev(s), _dev(r), _dev(w)
    L.check(eng.lib.xl_policy_forward(eng.handle, st.buf.data_ptr(), sd_.data_ptr(), rd.data_ptr(), wd.data_ptr(), None,
                                      B, Tn, so, L.XL_FLAG_DISCRETE if discrete else 0,
                                      torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert bool(torch.isnan(lp[2, 7, 0]))
    assert int(torch.isnan(lp).sum()) == 1
    # logprobs without targets: invalid argument
    so = C.byref(L.XLSeqOutputs(tokens=None, actions=None, logits=None, targets=None, logprobs=lp.data_ptr()))
    assert eng.lib.xl_policy_forward(eng.handle, st.buf.data_ptr(), sd_.data_ptr(), rd.data_ptr(), None, None, B, Tn,
                                     so, 0, torch.cuda.current_stream().cuda_stream) == L.XL_ERR_INVALID_ARG
    eng.close()


# ---- 5b: rejections through the raw ABI -------------------------------------------------------------------------------
def _raw_forward(eng, cache, s, r, lengths, tok, act, flags=0):
    B, Tn = s.shape[:2]
    so = L.XLSeqOutputs(tokens=tok.data_ptr(), actions=act.data_ptr(), logits=None, targets=None, logprobs=None)
    lens = None if lengths is None else np.ascontiguousarray(lengths, np.int32)
    return eng.lib.xl_policy_forward(eng.handle, cache.buf.data_ptr(), s.data_ptr(), r.data_ptr(), None,
                                     None if lens is None else lens.ctypes.data_as(C.c_void_p), B, Tn, C.byref(so),
                                     flags, torch.cuda.current_stream().cuda_stream)


@gpu
def test_policy_forward_rejections_leave_state_and_outputs_untouched():
    """XL_FLAG_STATE_EMBEDS, and ragged lengths on a shape without the sequence path (conv kernel 3): XL_ERR_UNSUPPORTED
    with state and outputs untouched. Uniform lengths on that shape take the step path, as the prefill does."""
    B, Tn = 3, 6
    for name, over, lengths, flags in (("16M", {}, None, L.XL_FLAG_STATE_EMBEDS),
                                       ("toy128", {"conv1d_kernel_size": 3}, [6, 0, 2], 0)):
        cfg, sd, eng = _engine(name, B, seed=14, **over)
        warm = _warm(eng, cfg, B, seed=15)
        s, r, _ = _inputs(cfg, B, Tn, seed=19)
        sd_, rd = _dev(s), _dev(r)
        cache = _copy(eng, warm)
        tok = torch.full((B, Tn, cfg.act_dim), 7, dtype=torch.int32, device="cuda")
        act = torch.full((B, Tn, cfg.act_dim), 5.0, device="cuda")
        assert _raw_forward(eng, cache, sd_, rd, lengths, tok, act, flags) == L.XL_ERR_UNSUPPORTED, name
        torch.cuda.synchronize()
        assert torch.equal(cache.buf, warm.buf), name
        assert bool((tok == 7).all() and (act == 5.0).all()), name
        if lengths is not None:
            a, b = _copy(eng, warm), _copy(eng, warm)
            oa = eng.policy_forward(a, sd_, rd, want_logits=True)
            ob = eng.policy_forward(b, sd_, rd, lengths=[Tn] * B, want_logits=True)
            torch.cuda.synchronize()
            assert torch.equal(a.buf, b.buf) and all(torch.equal(oa[k], ob[k]) for k in oa)
        eng.close()


# ---- 6: sampler and token ring ----------------------------------------------------------------------------------------
@gpu
def test_policy_forward_argmax_and_leaves_sampler_step_and_token_ring_alone():
    B, Tn = 4, 45
    cfg, sd, eng = _engine("16M", B, seed=10)
    s, r, w = _inputs(cfg, B, Tn + 1, seed=15)
    plain = eng.policy_forward(eng.new_state(B), _dev(s[:, :Tn]), _dev(r[:, :Tn]), _dev(w[:, :Tn]), want_logits=True)
    ring = torch.full((6, B, cfg.act_dim), -1, dtype=torch.int32, device="cuda")
    eng.set_token_ring(ring, next_slot=2)
    kw = dict(temperature=1.0, top_k=0, top_p=0.5, seed=1234)
    eng.set_sampling(**kw, step0=17)
    cache = eng.new_state(B)
    armed = eng.policy_forward(cache, _dev(s[:, :Tn]), _dev(r[:, :Tn]), _dev(w[:, :Tn]), want_logits=True)
    torch.cuda.synchronize()
    for k in plain:
        assert torch.equal(plain[k], armed[k]), k
    assert bool((ring == -1).all())
    out = eng.policy_step(cache, _dev(s[:, Tn]), _dev(r[:, Tn]), _dev(w[:, Tn]), want_logits=True)
    torch.cuda.synchronize()
    tok, _ = eng.sample_actions(out["action_logits"], step=17, **kw)
    assert torch.equal(out["action_tokens"], tok)
    assert torch.equal(ring[2], out["action_tokens"])
    assert bool((ring[[0, 1, 3, 4, 5]] == -1).all())
    eng.set_sampling(None)
    eng.set_token_ring(None)
    eng.close()


# ---- 7: Python layer --------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("discrete", [False, True])
def test_model_non_cache_forward(discrete):
    from lram_b200 import decision_xlstm as DX
    B, T = 3, 20
    cfg = preset("16M")
    sd = make_state_dict(cfg, seed=11)
    model = DX.MultiDomainDiscreteDecisionXLSTMModel(cfg, sd, max_batch=B)
    s, r, w = _inputs(cfg, B, T, seed=16)
    A = 1 if discrete else cfg.act_dim
    st, rt, rw = _dev(s), _dev(r).view(B, T, 1), _dev(w).view(B, T, 1)
    acts = torch.zeros(B, T, A, device="cuda")
    out = model(states=st, actions=acts, rewards=rw, returns_to_go=rt, timesteps=None,
                attention_mask=torch.zeros(B, T, device="cuda"), use_inference_cache=False)
    assert out.past_key_values is None and out.last_hidden_state is None
    assert tuple(out.action_preds.shape) == (B, T, A)
    assert tuple(out.action_logits.shape) == (B, T, A, cfg.num_actions)
    eng = model.engine
    ref = eng.policy_forward(eng.new_state(B), st, _dev(r), _dev(w), discrete=discrete, want_logits=True)
    torch.cuda.synchronize()
    assert torch.equal(out.action_logits.reshape(B, T, -1), ref["action_logits"])
    assert torch.equal(out.action_tokens, ref["action_tokens"].long())
    if discrete:
        assert torch.equal(out.action_preds, ref["action_tokens"][..., :1].long())
    else:
        assert torch.equal(out.action_preds, ref["action_preds"])
    # the last timestep equals the cache path stepped over the same T timesteps from zero
    pkv = None
    for t in range(T):
        o = model(states=st[:, :t + 1], actions=acts[:, :t + 1], rewards=rw[:, :t + 1], returns_to_go=rt[:, :t + 1],
                  timesteps=None, use_inference_cache=True, past_key_values=pkv)
        pkv = o.past_key_values
    torch.cuda.synchronize()
    _check_tokens(cfg, out.action_tokens[:, -1], o.action_logits[:, 0].cpu(), discrete, "model last timestep")
    assert _rel(out.action_logits[:, -1].cpu(), o.action_logits[:, 0].cpu()) < REL_TOL


@gpu
def test_encoder_non_cache_forward_vs_parallel_oracle():
    from lram_b200 import decision_xlstm as DX
    from oracle.xlstm_oracle import OracleEncoder
    cfg = preset("toy128")
    enc = DX.FusedXLSTMEncoder(config=cfg, max_batch=3).cuda()
    with torch.no_grad():
        for p in enc.parameters():                          # input-dependent gates (SURVEY.md §7)
            p.add_(torch.randn(p.shape, generator=torch.Generator().manual_seed(p.numel())).cuda() * 0.02)
    x = torch.randn(3, 90, cfg.d, generator=torch.Generator().manual_seed(3))
    out = enc(inputs_embeds=x.cuda(), use_cache=False)
    assert out.past_key_values is None
    sd = {"encoder." + k: v.cpu() for k, v in enc.state_dict().items()}
    ref = OracleEncoder(cfg, sd).forward_parallel(x)
    assert _rel(out.last_hidden_state.cpu(), ref) < REL_TOL


# ---- 8: large batch ---------------------------------------------------------------------------------------------------
@gpu
def test_policy_forward_large_batch_vs_graph_stepping():
    """Tokens equal to graph-replayed stepping of the same inputs. Both sides are the library, so the rule for a flip is
    the row's own evidence: the step's top-two margin must be below twice the largest logit difference of that row
    (the most a perturbation of that size can close). Flips are counted and printed."""
    B, Tn = 64, 300
    cfg, sd, eng = _engine("48M", B, seed=12)
    rng = np.random.default_rng(31)
    lengths = rng.integers(1, Tn + 1, B)
    lengths[:2] = [Tn, 1]
    s, r, w = _inputs(cfg, B, Tn, seed=17)
    out = eng.policy_forward(eng.new_state(B), _dev(s), _dev(r), _dev(w), lengths=lengths, want_logits=True)
    cache = eng.new_state(B)
    io = {"s": torch.empty(B, cfg.state_dim, device="cuda"), "r": torch.empty(B, device="cuda"),
          "w": torch.empty(B, device="cuda")}
    res = {"action_tokens": torch.zeros(B, cfg.act_dim, dtype=torch.int32, device="cuda"),
           "action_preds": torch.zeros(B, cfg.act_dim, device="cuda"),
           "action_logits": torch.empty(B, cfg.head_out, device="cuda")}
    tok, lgs = [], []
    sd_, rd, wd = _dev(s), _dev(r), _dev(w)
    for t in range(Tn):
        io["s"].copy_(sd_[:, t])
        io["r"].copy_(rd[:, t])
        io["w"].copy_(wd[:, t])
        eng.policy_step(cache, io["s"], io["r"], io["w"], flags=L.XL_FLAG_GRAPH, out=res)
        tok.append(res["action_tokens"].clone())
        lgs.append(res["action_logits"].view(B, cfg.act_dim, cfg.num_actions).clone())
    torch.cuda.synchronize()
    tok, lgs = torch.stack(tok, 1).cpu(), torch.stack(lgs, 1).cpu()
    fwd = out["action_logits"].cpu().view(B, Tn, cfg.act_dim, cfg.num_actions)
    flips = total = 0
    for b in range(B):
        n = int(lengths[b])
        assert _rel(fwd[b, :n], lgs[b, :n]) < REL_TOL, b
        top2 = lgs[b, :n].double().topk(2, dim=-1).values
        margin = top2[..., 0] - top2[..., 1]
        diff = (fwd[b, :n].double() - lgs[b, :n].double()).abs().amax(-1)
        fl = out["action_tokens"][b, :n].cpu() != tok[b, :n]
        for t, j in fl.nonzero().tolist():
            print(f"env {b} t {t} row {j}: flip at step margin {margin[t, j]:.3e}, row logit diff {diff[t, j]:.3e}")
        assert bool((margin[fl] < 2 * diff[fl]).all()), f"env {b}: token differs beyond the logit difference"
        flips += int(fl.sum())
        total += fl.numel()
    print(f"48M x {B} envs, lengths <= {Tn}: {flips} near-tie flips of {total} tokens")
    assert flips <= max(1, total // 1000)
    eng.close()


# ---- 9: the reference's own non-cache forward -------------------------------------------------------------------------
HERE = os.path.dirname(os.path.abspath(__file__))


def test_reference_non_cache_forward_vs_oracle():
    """The reference's `forward(use_inference_cache=False)` (through the stub packages and oracle/xlstm_shim.py) against
    the oracle stepping every timestep, the restatement the GPU tests above hold the library to."""
    sys.path.insert(0, os.path.join(HERE, "golden"))
    import ref_stubs
    if not ref_stubs.reference_available():
        pytest.skip(ref_stubs.SKIP_REASON)
    import make_ref_golden as G
    from oracle.xlstm_oracle import OraclePolicy
    cfg = preset("toy128")
    sd = make_state_dict(cfg, seed=13)
    policy = G.build_reference_policy(cfg, sd, with_image=False)
    B, T = 2, 6
    s, r, _ = _inputs(cfg, B, T, seed=18)
    with torch.no_grad():
        o = policy(states=torch.from_numpy(s), actions=torch.zeros(B, T, cfg.act_dim),
                   rewards=torch.zeros(B, T, 1), returns_to_go=torch.from_numpy(r).view(B, T, 1),
                   timesteps=torch.arange(T).repeat(B, 1), attention_mask=torch.ones(B, T, dtype=torch.long),
                   return_dict=True, deterministic=True, prompt=None, task_id=None, ddp_kwargs={},
                   use_inference_cache=False)
    ora, pkv, lg = OraclePolicy(cfg, sd), None, []
    for t in range(T):
        st = ora.step(torch.from_numpy(s[:, t]), torch.from_numpy(r[:, t]), past_key_values=pkv)
        pkv = st["past_key_values"]
        lg.append(st["action_logits"])
    ref = torch.stack(lg, 1)
    got = o.action_logits.reshape(B, T, cfg.act_dim, cfg.num_actions).float()
    assert _rel(got, ref) < REL_TOL
