"""Image observations on the sequence path: the context prefill and the sequence forward from state embeddings
(xl_policy_prefill_embeds / xl_policy_forward_embeds, `state_embeds=True` of XLSTMEngine.policy_prefill /
policy_forward), `image_encoder.embed_frames`, and the model's non-cache forward on frames and on `img_is_encoded`
embeddings. Checked against the oracle stepping each env, against the library's own policy steps and prefills, and at
the Python layer; the argument checks and embed_frames run without a GPU. Near-ties follow test_gpu_policy_forward.py."""
import ctypes as C

import numpy as np
import pytest
import torch

from lram_b200 import _lib as L
from lram_b200.config import preset
from lram_b200.image_encoder import ImpalaCNN, embed_frames, make_impala_state_dict, scale_frames, \
    split_image_weights

from test_gpu_policy_forward import (REL_TOL, _State, _check_tokens, _copy, _cpu, _dev, _engine, _env_pkv, _inputs,
                                     _nolib_engine, _rel, _shape_logits, _slots, _slots_equal)

gpu = pytest.mark.gpu


def _embeds(cfg, B, Tn, seed):
    """State embeddings [B, Tn, d] (numpy fp32) in the range of an ImpalaCNN output."""
    return np.abs(np.random.default_rng(seed).normal(0.0, 0.7, (B, Tn, cfg.d))).astype(np.float32)


# ---- CPU: argument checks and embed_frames --------------------------------------------------------------------------
def test_engine_state_embeds_arguments_rejected_before_the_library():
    eng = _nolib_engine("cpu")
    cfg, B, Tn = eng.cfg, 3, 8
    rtg = torch.zeros(B, Tn)
    for bad in (torch.zeros(B, Tn, cfg.state_dim), torch.zeros(B, Tn, cfg.d + 4), torch.zeros(B + 1, Tn, cfg.d),
                torch.zeros(B, cfg.d), torch.zeros(B, Tn, cfg.d, dtype=torch.float64),
                torch.zeros(B, Tn, cfg.d, dtype=torch.float16), np.zeros((B, Tn, cfg.d), np.float32)):
        with pytest.raises(ValueError):
            eng.policy_forward(_State(B), bad, rtg, state_embeds=True)
        with pytest.raises(ValueError):
            eng.policy_prefill(_State(B), bad, rtg, state_embeds=True)
    eng = _nolib_engine("cuda:0")                       # right shape and dtype, on the host
    ok = torch.zeros(B, Tn, cfg.d)
    with pytest.raises(ValueError):
        eng.policy_forward(_State(B), ok, rtg, state_embeds=True)
    with pytest.raises(ValueError):
        eng.policy_prefill(_State(B), ok, rtg, state_embeds=True)
    with pytest.raises(ValueError):                     # lengths are still checked
        eng.policy_forward(_State(B), ok, rtg, lengths=[1, 2])


def _cnn(d=32, seed=4):
    cnn = ImpalaCNN((3, 16, 16), d)
    cnn.load_state_dict(split_image_weights(make_impala_state_dict(d, (3, 16, 16), seed=seed)))
    return cnn.eval()


def test_embed_frames_sliced_equals_one_call():
    cnn = _cnn()
    B, T = 3, 7
    frames = torch.from_numpy(np.random.default_rng(1).integers(0, 256, (B, T, 3, 16, 16), dtype=np.uint8))
    ref = cnn(scale_frames(frames.reshape(B * T, 3, 16, 16))).view(B, T, -1)
    for m in (1, 4, 5, B * T, 1000):
        got = embed_frames(cnn, frames, max_frames=m)
        assert got.dtype == torch.float32 and tuple(got.shape) == (B, T, 32)
        torch.testing.assert_close(got, ref, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(embed_frames(cnn, frames.float(), max_frames=4), ref, rtol=1e-5, atol=1e-5)
    lens = [7, 0, 3]
    got = embed_frames(cnn, frames, lengths=lens, max_frames=2)
    for b, n in enumerate(lens):
        torch.testing.assert_close(got[b, :n], ref[b, :n], rtol=1e-5, atol=1e-5)
    for bad in ([1, 2], [8, 0, 0], [-1, 0, 0]):
        with pytest.raises(ValueError):
            embed_frames(cnn, frames, lengths=bad)
    with pytest.raises(ValueError):
        embed_frames(cnn, frames[:, :, :, :8])


def test_embed_frames_lengths_never_feed_frames_past_the_length():
    cnn = _cnn()
    B, T, lens = 3, 6, [6, 2, 0]
    frames = torch.from_numpy(np.random.default_rng(2).integers(0, 256, (B, T, 3, 16, 16))).float()
    for b, n in enumerate(lens):
        frames[b, n:] = float("nan")
    got = embed_frames(cnn, frames, lengths=lens, max_frames=4)
    assert not bool(torch.isnan(got).any())
    for b, n in enumerate(lens):
        assert bool((got[b, n:] == 0).all()), b
        if n:
            ref = cnn(scale_frames(frames[b, :n]))
            torch.testing.assert_close(got[b, :n], ref, rtol=1e-5, atol=1e-5)


# ---- GPU helpers ----------------------------------------------------------------------------------------------------
def _warm(eng, cfg, B, seed):
    """A non-zero start state: three embedding policy steps from zero."""
    e = _embeds(cfg, B, 3, seed + 1000)
    _, r, w = _inputs(cfg, B, 3, seed + 1000)
    cache = eng.new_state(B)
    for t in range(3):
        eng.policy_step(cache, _dev(e[:, t]), _dev(r[:, t]), _dev(w[:, t]), state_embeds=True)
    torch.cuda.synchronize()
    return cache


def _oracle(cfg, sd, pkv0, e, r, w):
    """OraclePolicy.step(state_embeds=True) over every timestep from pkv0 -> logits [B, Tn, act_dim, num_actions]."""
    from oracle.xlstm_oracle import OraclePolicy
    ora, pkv, lg = OraclePolicy(cfg, sd), pkv0, []
    for t in range(e.shape[1]):
        o = ora.step(torch.from_numpy(e[:, t]), torch.from_numpy(r[:, t]), torch.from_numpy(w[:, t]),
                     past_key_values=pkv, state_embeds=True)
        pkv = o["past_key_values"]
        lg.append(o["action_logits"])
    return torch.stack(lg, 1)


def _raw(eng, fn, cache, e, r, lengths=None, out=None, flags=0):
    """One raw-ABI sequence call; xl_policy_prefill is the one entry without a lengths argument."""
    B, Tn = e.shape[:2]
    lens = None if lengths is None else np.ascontiguousarray(lengths, np.int32)
    args = [eng.handle, cache.buf.data_ptr(), e.data_ptr(), r.data_ptr(), None]
    if fn is not eng.lib.xl_policy_prefill:
        args.append(None if lens is None else lens.ctypes.data_as(C.c_void_p))
    args += [B, Tn]
    if out is not None:
        args.append(C.byref(out))
    return fn(*args, flags, torch.cuda.current_stream().cuda_stream)


# ---- 1: against the oracle, state bytes equal to the prefill --------------------------------------------------------
_CASES = [("16M", (2, 1, 0)), ("toy128", (2, 1, 0)), ("toy128-ms", (2,)), ("48M-ms", (2,))]


@gpu
@pytest.mark.parametrize("name,cells", _CASES)
@pytest.mark.parametrize("Tn", [45, 200])
def test_forward_embeds_vs_oracle_every_cell(name, cells, Tn):
    B = 2
    cfg, sd, eng = _engine(name, B, seed=3)
    warm = _warm(eng, cfg, B, seed=5)
    e = _embeds(cfg, B, Tn, seed=11)
    _, r, w = _inputs(cfg, B, Tn, seed=11)
    ref_lg = _oracle(cfg, sd, _cpu(warm.to_past_key_values()), e, r, w)
    flips = 0
    for cell in cells:
        eng.set_option("prefill_cell", cell)
        pre = _copy(eng, warm)
        eng.policy_prefill(pre, _dev(e), _dev(r), _dev(w), state_embeds=True)
        for discrete in (False, True):
            cache = _copy(eng, warm)
            out = eng.policy_forward(cache, _dev(e), _dev(r), _dev(w), discrete=discrete, want_logits=True,
                                     state_embeds=True)
            torch.cuda.synchronize()
            assert torch.equal(cache.buf, pre.buf), (cell, discrete)        # bit-identical to the prefill
            lg = _shape_logits(cfg, out["action_logits"].cpu(), discrete)
            ref = ref_lg[:, :, :1] if discrete else ref_lg
            assert _rel(lg, ref) < REL_TOL, (cell, discrete)
            flips += _check_tokens(cfg, out["action_tokens"], ref, discrete, f"{name} cell {cell} d={discrete}")
            if discrete:
                assert bool((out["action_tokens"][..., 1:] == -1).all() and (out["action_preds"][..., 1:] == 0).all())
    eng.set_option("prefill_cell", 2)
    print(f"{name} Tn={Tn}: {flips} near-tie flips")
    eng.close()


# ---- 2: all tail: bit-identical to embedding policy steps -----------------------------------------------------------
@gpu
@pytest.mark.parametrize("discrete", [False, True])
def test_forward_embeds_short_equals_eager_steps(discrete):
    B, Tn = 3, 5
    cfg, sd, eng = _engine("16M", B, seed=4)
    warm = _warm(eng, cfg, B, seed=6)
    e = _embeds(cfg, B, Tn, seed=12)
    _, r, w = _inputs(cfg, B, Tn, seed=12)
    cache = _copy(eng, warm)
    out = eng.policy_forward(cache, _dev(e), _dev(r), _dev(w), discrete=discrete, want_logits=True, state_embeds=True)
    pre = _copy(eng, warm)
    eng.policy_prefill(pre, _dev(e), _dev(r), _dev(w), state_embeds=True)
    step = _copy(eng, warm)
    flags = L.XL_FLAG_DISCRETE if discrete else 0
    for t in range(Tn):
        o = eng.policy_step(step, _dev(e[:, t]), _dev(r[:, t]), _dev(w[:, t]), flags=flags, want_logits=True,
                            state_embeds=True)
        torch.cuda.synchronize()
        cols = slice(0, 1) if discrete else slice(None)
        assert torch.equal(out["action_tokens"][:, t, cols], o["action_tokens"][:, cols]), t
        assert torch.equal(out["action_preds"][:, t, cols], o["action_preds"][:, cols]), t
        assert torch.equal(out["action_logits"][:, t], o["action_logits"]), t
    assert torch.equal(cache.buf, step.buf) and torch.equal(pre.buf, step.buf)
    eng.close()


# ---- 3 + 4: ragged lengths ------------------------------------------------------------------------------------------
@gpu
def test_forward_embeds_ragged():
    B, Tn, lengths = 6, 200, [200, 0, 45, 7, 133, 45]
    cfg, sd, eng = _engine("16M", B, seed=7)
    warm = _warm(eng, cfg, B, seed=8)
    e = _embeds(cfg, B, Tn, seed=13)
    _, r, w = _inputs(cfg, B, Tn, seed=13)
    en, rn, wn = e.copy(), r.copy(), w.copy()
    for b, n in enumerate(lengths):                     # never read
        en[b, n:], rn[b, n:], wn[b, n:] = np.nan, np.nan, np.nan
    tg = torch.randint(-1, cfg.num_actions, (B, Tn, cfg.act_dim), generator=torch.Generator().manual_seed(1)).cuda()
    cache = _copy(eng, warm)
    out = eng.policy_forward(cache, _dev(en), _dev(rn), _dev(wn), lengths=lengths, targets=tg, want_logits=True,
                             state_embeds=True)
    pre = _copy(eng, warm)
    eng.policy_prefill(pre, _dev(en), _dev(rn), _dev(wn), lengths=lengths, state_embeds=True)
    torch.cuda.synchronize()
    assert torch.equal(cache.buf, pre.buf)                                     # == the ragged prefill
    assert _slots_equal(_slots(cfg, cache, 1), _slots(cfg, warm, 1))           # length 0: untouched
    for b, n in enumerate(lengths):
        assert bool((out["action_tokens"][b, n:] == -1).all()), b
        for k in ("action_preds", "action_logits", "action_logprobs"):
            assert bool((out[k][b, n:] == 0).all()), (b, k)
        assert not bool(torch.isnan(out["action_logits"][b]).any()), b
    # each env against its own uniform forward (B = 1)
    wpkv = warm.to_past_key_values()
    for b, n in enumerate(lengths):
        if not n:
            continue
        one = eng.new_state(1)
        one.load_past_key_values(_env_pkv(wpkv, b))
        o1 = eng.policy_forward(one, _dev(e[b:b + 1, :n]), _dev(r[b:b + 1, :n]), _dev(w[b:b + 1, :n]),
                                targets=tg[b:b + 1, :n].contiguous(), want_logits=True, state_embeds=True)
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
    os_ = eng.policy_forward(cs, _dev(en[perm]), _dev(rn[perm]), _dev(wn[perm]), lengths=[lengths[b] for b in perm],
                             targets=tg[perm].contiguous(), want_logits=True, state_embeds=True)
    torch.cuda.synchronize()
    for k, b in enumerate(perm):
        for key in out:
            assert torch.equal(os_[key][k], out[key][b]), (k, b, key)
        assert _slots_equal(_slots(cfg, cs, k), _slots(cfg, cache, b)), (k, b)
    # lengths all Tn: the uniform call, bit for bit (forward and prefill)
    a, c = _copy(eng, warm), _copy(eng, warm)
    oa = eng.policy_forward(a, _dev(e), _dev(r), _dev(w), want_logits=True, state_embeds=True)
    oc = eng.policy_forward(c, _dev(e), _dev(r), _dev(w), lengths=[Tn] * B, want_logits=True, state_embeds=True)
    pa, pc = _copy(eng, warm), _copy(eng, warm)
    eng.policy_prefill(pa, _dev(e), _dev(r), _dev(w), state_embeds=True)
    eng.policy_prefill(pc, _dev(e), _dev(r), _dev(w), lengths=[Tn] * B, state_embeds=True)
    torch.cuda.synchronize()
    assert torch.equal(a.buf, c.buf) and all(torch.equal(oa[k], oc[k]) for k in oa)
    assert torch.equal(pa.buf, pc.buf) and torch.equal(pa.buf, a.buf)
    eng.close()


# ---- 5: log-probabilities -------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("discrete", [False, True])
def test_forward_embeds_logprobs(discrete):
    B, Tn = 3, 61
    cfg, sd, eng = _engine("16M", B, seed=9)
    e = _embeds(cfg, B, Tn, seed=14)
    _, r, w = _inputs(cfg, B, Tn, seed=14)
    tg = torch.randint(0, cfg.num_actions, (B, Tn, cfg.act_dim), generator=torch.Generator().manual_seed(2))
    tg[0, :, 5:] = -1
    tg = tg.cuda()
    out = eng.policy_forward(eng.new_state(B), _dev(e), _dev(r), _dev(w), discrete=discrete, targets=tg,
                             want_logits=True, state_embeds=True)
    torch.cuda.synchronize()
    lg = _shape_logits(cfg, out["action_logits"].cpu(), discrete).double()
    ls = torch.log_softmax(lg, dim=-1)
    t = tg.cpu().long()
    cols = 1 if discrete else cfg.act_dim
    exp = ls.gather(-1, t[..., :cols].clamp(min=0).unsqueeze(-1)).squeeze(-1)
    exp = torch.where(t[..., :cols] < 0, torch.zeros_like(exp), exp)
    got = out["action_logprobs"].cpu().double()
    assert (got[..., :cols] - exp).abs().max().item() < 1e-5
    if discrete:
        assert bool((got[..., 1:] == 0).all())
    eng.close()


# ---- 6: rejections ----------------------------------------------------------------------------------------------------
@gpu
def test_embeds_rejections_leave_state_untouched():
    B, Tn = 3, 20
    cfg, sd, eng = _engine("16M", B, seed=14)
    warm = _warm(eng, cfg, B, seed=15)
    s, r, _ = _inputs(cfg, B, Tn, seed=19)
    e = _dev(_embeds(cfg, B, Tn, seed=19))
    sd_, rd = _dev(s), _dev(r)
    cache = _copy(eng, warm)
    # raw-state prefills refuse state embeddings (they would read them as [B, Tn, state_dim])
    for lengths in (None, [20, 0, 7]):
        fn = eng.lib.xl_policy_prefill_ragged if lengths else eng.lib.xl_policy_prefill
        assert _raw(eng, fn, cache, e, rd, lengths, flags=L.XL_FLAG_STATE_EMBEDS) == L.XL_ERR_UNSUPPORTED
        assert "_embeds" in eng.lib.xl_last_error().decode()
    # a misaligned embedding pointer, and logprobs without targets: invalid arguments
    flat = torch.zeros(B * Tn * cfg.d + 1, device="cuda")
    mis = flat[1:].view(B, Tn, cfg.d)
    tok = torch.full((B, Tn, cfg.act_dim), 7, dtype=torch.int32, device="cuda")
    lp = torch.full((B, Tn, cfg.act_dim), 5.0, device="cuda")
    so = L.XLSeqOutputs(tokens=tok.data_ptr(), actions=None, logits=None, targets=None, logprobs=None)
    assert _raw(eng, eng.lib.xl_policy_prefill_embeds, cache, mis, rd) == L.XL_ERR_INVALID_ARG
    assert _raw(eng, eng.lib.xl_policy_forward_embeds, cache, mis, rd, out=so) == L.XL_ERR_INVALID_ARG
    so = L.XLSeqOutputs(tokens=tok.data_ptr(), actions=None, logits=None, targets=None, logprobs=lp.data_ptr())
    assert _raw(eng, eng.lib.xl_policy_forward_embeds, cache, e, rd, out=so) == L.XL_ERR_INVALID_ARG
    torch.cuda.synchronize()
    assert torch.equal(cache.buf, warm.buf)
    assert bool((tok == 7).all() and (lp == 5.0).all())
    # the Python layer copies a misaligned view instead of failing
    a, b = _copy(eng, warm), _copy(eng, warm)
    mis.copy_(e)
    eng.policy_prefill(a, mis, rd, state_embeds=True)
    eng.policy_prefill(b, e, rd, state_embeds=True)
    torch.cuda.synchronize()
    assert torch.equal(a.buf, b.buf)
    # XL_FLAG_STATE_EMBEDS on the _embeds entries is redundant
    c = _copy(eng, warm)
    assert _raw(eng, eng.lib.xl_policy_prefill_embeds, c, e, rd, flags=L.XL_FLAG_STATE_EMBEDS) == L.XL_OK
    torch.cuda.synchronize()
    assert torch.equal(c.buf, b.buf)
    eng.close()


# ---- 7: sampler and token ring ----------------------------------------------------------------------------------------
@gpu
def test_forward_embeds_argmax_and_leaves_sampler_step_and_token_ring_alone():
    B, Tn = 4, 45
    cfg, sd, eng = _engine("16M", B, seed=10)
    e = _embeds(cfg, B, Tn + 1, seed=15)
    _, r, w = _inputs(cfg, B, Tn + 1, seed=15)
    E, R, W = _dev(e[:, :Tn]), _dev(r[:, :Tn]), _dev(w[:, :Tn])
    plain = eng.policy_forward(eng.new_state(B), E, R, W, want_logits=True, state_embeds=True)
    ring = torch.full((6, B, cfg.act_dim), -1, dtype=torch.int32, device="cuda")
    eng.set_token_ring(ring, next_slot=2)
    kw = dict(temperature=1.0, top_k=0, top_p=0.5, seed=1234)
    eng.set_sampling(**kw, step0=17)
    cache = eng.new_state(B)
    eng.policy_prefill(eng.new_state(B), E, R, W, state_embeds=True)
    armed = eng.policy_forward(cache, E, R, W, want_logits=True, state_embeds=True)
    torch.cuda.synchronize()
    for k in plain:
        assert torch.equal(plain[k], armed[k]), k
    assert bool((ring == -1).all())
    out = eng.policy_step(cache, _dev(e[:, Tn]), _dev(r[:, Tn]), _dev(w[:, Tn]), want_logits=True, state_embeds=True)
    torch.cuda.synchronize()
    tok, _ = eng.sample_actions(out["action_logits"], step=17, **kw)
    assert torch.equal(out["action_tokens"], tok)
    assert torch.equal(ring[2], out["action_tokens"])
    assert bool((ring[[0, 1, 3, 4, 5]] == -1).all())
    eng.set_sampling(None)
    eng.set_token_ring(None)
    eng.close()


# ---- 8: the model end to end ------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("discrete", [False, True])
def test_model_image_sequence_forward_vs_oracle(discrete):
    from lram_b200.decision_xlstm import MultiDomainDiscreteDecisionXLSTMModel
    from lram_b200.synth import make_state_dict
    from oracle.xlstm_oracle import OraclePolicy
    cfg = preset("toy128")
    sd = make_state_dict(cfg, seed=0)
    sd.update(make_impala_state_dict(cfg.d, (3, 64, 64), seed=9))
    B, T = 3, 21
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        model = MultiDomainDiscreteDecisionXLSTMModel(cfg, sd, max_batch=B)
        model.image_max_frames = 16                 # several CNN slices
        frames = torch.from_numpy(np.random.default_rng(3).integers(0, 256, (B, T, 3, 64, 64), dtype=np.uint8))
        rtg = torch.linspace(5.0, 3.0, T).repeat(B, 1).view(B, T, 1)
        act = torch.zeros(B, T, 1, dtype=torch.long) if discrete else torch.zeros(B, T, cfg.act_dim)
        out = model(states=frames, actions=act, rewards=None, returns_to_go=rtg, use_inference_cache=False)
        A = 1 if discrete else cfg.act_dim
        assert out.past_key_values is None and tuple(out.action_logits.shape) == (B, T, A, cfg.num_actions)
        ora, pkv, lg = OraclePolicy(cfg, sd), None, []
        for t in range(T):
            o = ora.step(frames[:, t], rtg[:, t].view(B), past_key_values=pkv, discrete=discrete)
            pkv = o["past_key_values"]
            lg.append(o["action_logits"])
        ref = torch.stack(lg, 1)[:, :, :A]
        assert _rel(out.action_logits.cpu(), ref) < REL_TOL
        _check_tokens(cfg, out.action_tokens.int(), ref, discrete, f"model frames d={discrete}")
        # img_is_encoded: [B, T, d] embeddings through the same call, bit-identical to the engine's forward
        emb = embed_frames(model.embed_image, frames)
        model.img_is_encoded = True
        enc = model(states=emb, actions=act, rewards=None, returns_to_go=rtg, use_inference_cache=False)
        eng = model.engine
        direct = eng.policy_forward(eng.new_state(B), emb, rtg.view(B, T).cuda(), discrete=discrete, want_logits=True,
                                    state_embeds=True)
        torch.cuda.synchronize()
        assert torch.equal(enc.action_logits.reshape(B, T, -1), direct["action_logits"])
        assert torch.equal(enc.action_tokens, direct["action_tokens"].long())
        model.engine.close()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
