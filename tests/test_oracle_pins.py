"""CPU tests: pin the oracle (SURVEY.md §4 i-iv / §8c) and the host-side tokenizers against golden vectors."""
import math
import os

import numpy as np
import pytest
import torch

from lram_b200.config import preset
from lram_b200.synth import make_state_dict, make_stream
from lram_b200 import tokenizers as T
from oracle import xlstm_oracle as O


def _npz(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


# ---- (iv) tokenizer known answers produced by the reference's own code ------------------------------------
def test_tokenizer_inline_kat():
    # SURVEY.md §4 (iv): values printed by src/tokenizers_custom/minmax_tokenizer.py in the build container
    x = torch.tensor([[-1, -0.999, 0, 0.5, 0.9999, 1, 1.5, -2]], dtype=torch.float32)
    for cls in (T.MinMaxTokenizer, ):
        tok = cls(vocab_size=256, shift=18)
        t = tok.tokenize(x)
        assert t.tolist() == [[18, 18, 146, 210, 273, 273, 273, 18]]
        assert tok.inv_tokenize(t).tolist() == [[-1, -1, 0, 0.5, 0.9921875, 0.9921875, 0.9921875, -1]]
        assert cls(vocab_size=64).tokenize(x).tolist() == [[0, 0, 32, 48, 63, 63, 63, 0]]
    o = O.OracleMinMaxTokenizer(256, 18)
    assert o.tokenize(x).tolist() == [[18, 18, 146, 210, 273, 273, 273, 18]]


@pytest.mark.parametrize("tag,vocab,shift", [("mm256s18", 256, 18), ("mm64s0", 64, 0), ("mm100s0", 100, 0)])
def test_minmax_tokenizer_golden(golden_dir, tag, vocab, shift):
    g = _npz(golden_dir, "tokenizer_kat.npz")
    x = torch.from_numpy(g["x"])
    for tok in (T.MinMaxTokenizer(vocab_size=vocab, shift=shift), O.OracleMinMaxTokenizer(vocab, shift)):
        t = tok.tokenize(x.clone())
        assert np.array_equal(t.numpy(), g[f"{tag}_tok"])                       # integer: bit exact
        assert np.array_equal(tok.inv_tokenize(t.clone()).numpy(), g[f"{tag}_inv"])


def test_minmax_inverse_all_ids(golden_dir):
    g = _npz(golden_dir, "tokenizer_kat.npz")
    ids = torch.arange(0, 274).view(1, -1)
    for tok in (T.MinMaxTokenizer(vocab_size=256, shift=18), O.OracleMinMaxTokenizer(256, 18)):
        assert np.array_equal(tok.inv_tokenize(ids.clone()).numpy(), g["mm256s18_inv_all_ids"])
    assert (g["mm256s18_inv_all_ids"][0, :18] == -1.0).all()                    # Appendix C.4


def test_minmax2_and_mulaw_golden(golden_dir):
    g = _npz(golden_dir, "tokenizer_kat.npz")
    x = torch.from_numpy(g["x"])
    t2 = T.MinMaxTokenizer2(vocab_size=256, shift=18)
    tok = t2.tokenize(x.clone())
    assert np.array_equal(tok.numpy(), g["mm2_256s18_tok"])
    assert np.array_equal(t2.inv_tokenize(tok.clone()).numpy(), g["mm2_256s18_inv"])
    mu = T.MuLawTokenizer(vocab_size=256, shift=0)
    xm = torch.from_numpy(g["mulaw_x"])
    tm = mu.tokenize(xm.clone())
    assert np.array_equal(tm.numpy(), g["mulaw256_tok"])
    np.testing.assert_allclose(mu.inv_tokenize(tm.clone()).numpy(), g["mulaw256_inv"], rtol=1e-6, atol=1e-7)
    # numpy branch of the reference
    tn = mu.tokenize(g["mulaw_x"].astype(np.float64))
    assert np.abs(tn - g["mulaw256_tok"]).max() <= 1


def test_make_tokenizer_factory():
    assert isinstance(T.make_tokenizer("minmax", {"vocab_size": 8}), T.MinMaxTokenizer)
    assert isinstance(T.make_tokenizer("minmax2"), T.MinMaxTokenizer2)
    assert isinstance(T.make_tokenizer("mulaw"), T.MuLawTokenizer)
    with pytest.raises(ValueError):
        T.make_tokenizer("nope")


# ---- (i) the cell step vs the independent HF implementation ------------------------------------------------
def test_cell_step_matches_hf_native(golden_dir):
    g = _npz(golden_dir, "hf_mlstm_step.npz")
    q, k, v, ig, fg = (torch.from_numpy(g[n]) for n in ("q", "k", "v", "ig", "fg"))
    Tn, B, NH, DH = q.shape
    c = torch.zeros(B, NH, DH, DH)
    n = torch.zeros(B, NH, DH, 1)
    m = torch.zeros(B, NH, 1, 1)
    for t in range(Tn):
        h, (c, n, m) = O.recurrent_step_stabilized_simple(
            c, n, m, q[t].unsqueeze(2), k[t].unsqueeze(2), v[t].unsqueeze(2), ig[t].unsqueeze(-1), fg[t].unsqueeze(-1))
        np.testing.assert_allclose(h.squeeze(2).numpy(), g["h"][t], rtol=2e-4, atol=2e-5)
    s = math.sqrt(DH)
    np.testing.assert_allclose((c * s).numpy(), g["c_final"], rtol=1e-4, atol=1e-5)   # C_hf = sqrt(DH) C
    np.testing.assert_allclose((n.squeeze(-1) * s).numpy(), g["n_final"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(m.view(B, NH, 1).numpy(), g["m_final"], rtol=0, atol=1e-6)


def test_recurrence_from_nonzero_state_matches_hf_chunkwise(golden_dir):
    """48 oracle steps from a NON-ZERO (C, n, m) == transformers' chunkwise-parallel forward (chunk 16) started from the
    same state: pins the recurrence over a sequence, the stabiliser carry and the state hand-over (prefill <-> stepping)."""
    g = _npz(golden_dir, "hf_mlstm_chunkwise.npz")
    q, k, v, ig, fg = (torch.from_numpy(g[n]) for n in ("q", "k", "v", "ig", "fg"))
    B, NH, S, DH = q.shape
    s = math.sqrt(DH)
    c = torch.from_numpy(g["c0"]) / s                       # C_hf = sqrt(DH) C (q scaled instead of k)
    n = (torch.from_numpy(g["n0"]) / s).unsqueeze(-1)
    m = torch.from_numpy(g["m0"]).unsqueeze(-1)
    for t in range(S):
        h, (c, n, m) = O.recurrent_step_stabilized_simple(
            c, n, m, q[:, :, t:t + 1], k[:, :, t:t + 1], v[:, :, t:t + 1], ig[:, :, t].view(B, NH, 1, 1),
            fg[:, :, t].view(B, NH, 1, 1))
        np.testing.assert_allclose(h.squeeze(2).numpy(), g["h"][:, :, t], rtol=5e-4, atol=1e-4)
    np.testing.assert_allclose((c * s).numpy(), g["c_final"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose((n.squeeze(-1) * s).numpy(), g["n_final"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(m.view(B, NH, 1).numpy(), g["m_final"], rtol=0, atol=1e-5)


def test_multihead_layer_norm_matches_hf(golden_dir):
    """oracle MultiHeadLayerNorm (group_norm, gamma = 1 + w) == transformers' xLSTMMultiHeadLayerNorm with weight 1 + w."""
    g = _npz(golden_dir, "hf_mlstm_chunkwise.npz")
    x = torch.from_numpy(g["ln_x"])                         # [B, S, NH, DH]
    B, S, NH, DH = x.shape
    y = O.multihead_layer_norm(x.permute(0, 2, 1, 3).contiguous(), torch.from_numpy(g["ln_w_residual"]), eps=1e-5)
    np.testing.assert_allclose(y.permute(0, 2, 1, 3).reshape(B, S, NH * DH).numpy(), g["ln_y"], rtol=1e-5, atol=2e-6)


# ---- (ii) recurrent == parallel -----------------------------------------------------------------------------
@pytest.mark.parametrize("name,S", [("toy", 24), ("toy128", 9)])
def test_recurrent_equals_parallel(name, S):
    cfg = preset(name)
    enc = O.OracleEncoder(cfg, make_state_dict(cfg, seed=3))
    x = torch.randn(2, S, cfg.d, generator=torch.Generator().manual_seed(5))
    y_rec, _ = enc.forward_cached(x, None)
    y_par = enc.forward_parallel(x)
    assert (y_rec - y_par).abs().max().item() < 2e-5


# ---- (iii) parameter counts vs README names ------------------------------------------------------------------
@pytest.mark.parametrize("name,enc_m,bytes_tok", [("16M", 12.94, 16974080), ("48M", 43.27, 57065856),
                                                   ("110M", 102.09, 135004672), ("206M", 198.84, 263373440)])
def test_param_counts_and_bytes(name, enc_m, bytes_tok):
    cfg = preset(name)
    assert abs(cfg.encoder_params() / 1e6 - enc_m) < 0.01
    assert cfg.algorithmic_bytes_per_env_layer_tokenstep() * cfg.num_blocks == bytes_tok   # SURVEY §8 table
    sd = make_state_dict(cfg, seed=0) if name == "16M" else None
    if sd is not None:
        n_enc = sum(v.numel() for k, v in sd.items() if k.startswith("encoder."))
        assert n_enc == cfg.encoder_params()


# ---- regression: committed oracle outputs ---------------------------------------------------------------------
@pytest.mark.parametrize("name", ["toy", "toy128"])
def test_oracle_regression(golden_dir, name):
    g = _npz(golden_dir, "oracle_toy.npz")
    cfg = preset(name)
    pol = O.OraclePolicy(cfg, make_state_dict(cfg, seed=0))
    states, rtg = g[f"{name}_states"], g[f"{name}_rtg"]
    st2, rtg2, _ = make_stream(cfg, range(states.shape[1]), states.shape[0], domains="mixed", seed=1234)
    assert np.array_equal(states, st2) and np.array_equal(rtg, rtg2)            # stream generator is stable
    pkv = None
    for t in range(states.shape[0]):
        o = pol.step(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), past_key_values=pkv)
        pkv = o["past_key_values"]
        assert np.array_equal(o["action_tokens"].numpy(), g[f"{name}_tokens"][t])
        np.testing.assert_allclose(o["last_hidden_state"].numpy(), g[f"{name}_hidden"][t], rtol=1e-4, atol=1e-5)
        assert np.array_equal(o["action_preds"].numpy(), g[f"{name}_actions"][t])


# ---- batch rows are independent (inf_dummy_batch_size trick relies on it) -------------------------------------
def test_batched_equals_single_env():
    cfg = preset("toy")
    pol = O.OraclePolicy(cfg, make_state_dict(cfg, seed=0))
    states, rtg, _ = make_stream(cfg, range(4), 3, domains="mixed")
    pkv = None
    singles = [None] * 4
    for t in range(3):
        ob = pol.step(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), past_key_values=pkv)
        pkv = ob["past_key_values"]
        for e in range(4):
            o1 = pol.step(torch.from_numpy(states[t, e:e + 1]), torch.from_numpy(rtg[t, e:e + 1]),
                          past_key_values=singles[e])
            singles[e] = o1["past_key_values"]
            assert torch.equal(o1["action_tokens"][0], ob["action_tokens"][e])
            assert (o1["last_hidden_state"][0] - ob["last_hidden_state"][e]).abs().max() < 1e-5


def test_reset_rows_equals_none_state():
    cfg = preset("toy")
    pol = O.OraclePolicy(cfg, make_state_dict(cfg, seed=0))
    states, rtg, _ = make_stream(cfg, range(3), 3, domains="mixed")
    pkv = None
    for t in range(2):
        pkv = pol.step(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), past_key_values=pkv)["past_key_values"]
    mask = torch.tensor([False, True, False])
    o = pol.step(torch.from_numpy(states[2]), torch.from_numpy(rtg[2]), past_key_values=O.reset_state_rows(pkv, mask))
    # a fresh batch of the same size: CPU BLAS picks its GEMM kernels by shape and host ISA, so a batch of another size
    # may round differently (batch-size independence is test_batched_equals_single_env's pin)
    fresh = pol.step(torch.from_numpy(states[2]), torch.from_numpy(rtg[2]), past_key_values=None)
    assert torch.equal(o["action_tokens"][1], fresh["action_tokens"][1])
    assert (o["last_hidden_state"][1] - fresh["last_hidden_state"][1]).abs().max() < 1e-6


def test_discrete_head_branch():
    cfg = preset("toy")
    pol = O.OraclePolicy(cfg, make_state_dict(cfg, seed=0))
    states, rtg, _ = make_stream(cfg, range(3), 1)
    o = pol.step(torch.from_numpy(states[0]), torch.from_numpy(rtg[0]), discrete=True)
    assert o["action_tokens"].shape == (3, 1) and int(o["action_tokens"].max()) < cfg.discrete_actions
    assert o["action_logits"].shape == (3, 1, cfg.num_actions)


# ---- sLSTM block (xLSTM[7:1] stacks): no external vectors exist ("parity unpinned"); internal pins only -------
def test_slstm_first_step_closed_form():
    """From the zero state the sLSTM update has a closed form: m' = i~ (n == 0 branch), i = 1, f = min(exp(logsig(f~)
    - i~), 1), c' = tanh(z~), n' = 1, y' = sigmoid(o~) tanh(z~) — checks gate order (i, f, z, o) and the branch."""
    from oracle.xlstm_oracle import slstm_pointwise
    g = torch.Generator().manual_seed(3)
    raw = torch.randn(5, 4, 16, generator=g)
    st = slstm_pointwise(raw, torch.zeros(4, 5, 16))
    assert torch.allclose(st[3], raw[:, 0])
    assert torch.allclose(st[1], torch.tanh(raw[:, 2]), atol=1e-7)
    assert torch.allclose(st[2], torch.ones(5, 16))
    assert torch.allclose(st[0], torch.sigmoid(raw[:, 3]) * torch.tanh(raw[:, 2]), atol=1e-7)
    # second step: stabilised form == unstabilised exponential-gate recurrence (eqs. 8-17) where that is finite
    raw2 = torch.randn(5, 4, 16, generator=g)
    st2 = slstm_pointwise(raw2, st)
    i1, i2 = torch.exp(raw[:, 0].double()), torch.exp(raw2[:, 0].double())
    f2 = torch.sigmoid(raw2[:, 1].double())
    c_true = f2 * (i1 * torch.tanh(raw[:, 2].double())) + i2 * torch.tanh(raw2[:, 2].double())
    n_true = f2 * i1 + i2
    y_true = torch.sigmoid(raw2[:, 3].double()) * c_true / n_true
    assert torch.allclose(st2[0].double(), y_true, atol=1e-5)
    # the stabiliser only rescales c and n by exp(-m)
    assert torch.allclose((st2[1] * torch.exp(st2[3])).double(), c_true, rtol=1e-4, atol=1e-5)


def test_slstm_stack_batched_equals_single_env_and_reset():
    from oracle.xlstm_oracle import OraclePolicy, reset_state_rows
    cfg = preset("toy128-ms")
    sd = make_state_dict(cfg, seed=2)
    pol = OraclePolicy(cfg, sd)
    states, rtg, _ = make_stream(cfg, range(3), 4, domains="mixed")
    pkv, single = None, [None] * 3
    for t in range(3):
        o = pol.step(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), past_key_values=pkv)
        pkv = o["past_key_values"]
        for b in range(3):
            ob = pol.step(torch.from_numpy(states[t, b:b + 1]), torch.from_numpy(rtg[t, b:b + 1]),
                          past_key_values=single[b])
            single[b] = ob["past_key_values"]
            assert torch.equal(ob["action_tokens"][0], o["action_tokens"][b])
            assert torch.allclose(ob["last_hidden_state"][0], o["last_hidden_state"][b], atol=2e-5)
    assert set(pkv["block_0"]) == {"slstm_state", "conv_state"} and pkv["block_0"]["slstm_state"].shape == (4, 3, cfg.d)
    assert set(pkv["block_1"]) == {"mlstm_state", "conv_state"}
    # reset of env 1 == env 1 starting from None
    r = reset_state_rows(pkv, torch.tensor([False, True, False]))
    o = pol.step(torch.from_numpy(states[3]), torch.from_numpy(rtg[3]), past_key_values=r)
    f = pol.step(torch.from_numpy(states[3, 1:2]), torch.from_numpy(rtg[3, 1:2]), past_key_values=None)
    assert torch.allclose(o["last_hidden_state"][1], f["last_hidden_state"][0], atol=2e-5)


def test_slstm_param_count():
    """xlstm_ms_mediumplus (d=768, 12 blocks, sLSTM at 1): per sLSTM block 2 d^2 (gates + recurrent kernel) +
    3 * 1024 * d (feed-forward) + small terms."""
    cfg = preset("48M-ms")
    sd = make_state_dict(preset("toy-ms"), seed=0)
    toy = preset("toy-ms")
    n_enc = sum(v.numel() for k, v in sd.items() if k.startswith("encoder."))
    assert n_enc == toy.encoder_params()
    assert cfg.ffn_dim == 1024 and preset("206M", slstm_at=(1,)).ffn_dim == 1664
    d = 768
    per_slstm = 2 * d * d + 3 * 1024 * d + d * 4 + d + 4 * d + 3 * d
    assert cfg.encoder_params() == 11 * (preset("48M").encoder_params() - d) // 12 + per_slstm + d
