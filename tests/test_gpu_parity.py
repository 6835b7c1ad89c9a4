"""GPU parity tests (run on the B200 box: python -m pytest tests -m gpu). Everything goes through the C-ABI
library; the oracle (oracle/xlstm_oracle.py) and the committed golden vectors are only the checker.

Tolerances (BASELINE.json north_star): action tokens / argmax actions bit-exact; hidden states and
continuous actions within 1e-3 relative of the fp32 oracle.
"""
import math
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from lram_b200 import _lib as L  # noqa: E402
from lram_b200.config import preset  # noqa: E402
from lram_b200.synth import make_state_dict, make_stream  # noqa: E402

REL_TOL = 1e-3
DEFAULT_SCAN_SPLIT = 2      # library default of xl_set_option("prefill_scan_split")


def _engine(name, B, seed=0, **over):
    from lram_b200.engine import XLSTMEngine
    cfg = preset(name, **over)
    sd = make_state_dict(cfg, seed=seed)
    return cfg, sd, XLSTMEngine(cfg, sd, max_batch=B)


def _rel(a, b):
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _margin_ok(ref_logits, tok_gpu, tok_ref):
    """Where tokens differ, report the oracle's top-2 margin (SURVEY §7 hard parts). Returns list of margins."""
    bad = (tok_gpu != tok_ref).nonzero()
    out = []
    for idx in bad:
        lg = ref_logits[tuple(idx.tolist())]
        top2 = torch.topk(lg, 2).values
        out.append(((top2[0] - top2[1]) / top2[0].abs().clamp_min(1e-30)).item())
    return out


# ------------------------------------------------------------------------------------------------------------
# unit: the cell kernel alone
# ------------------------------------------------------------------------------------------------------------
def test_cell_step_vs_hf_golden(golden_dir):
    """recurrent step kernel vs vectors from transformers' mlstm_recurrent_step_native (independent impl)."""
    g = np.load(os.path.join(golden_dir, "hf_mlstm_step.npz"))
    Tn, B, NH, DH = g["q"].shape
    cfg, sd, eng = _engine("toy", B)            # toy: NH=4, DH=32, inner=128
    assert (cfg.num_heads, cfg.head_dim) == (NH, DH)
    dev = eng.device
    C = torch.zeros(B, NH, DH, DH, device=dev)
    n = torch.zeros(B, NH, DH, device=dev)
    m = torch.zeros(B, NH, device=dev)
    w0 = torch.zeros(cfg.inner, device=dev)
    for t in range(Tn):
        qkv = torch.stack([torch.from_numpy(g[k][t]).reshape(B, NH * DH) for k in ("q", "k", "v")], dim=1).to(dev)
        ig = torch.from_numpy(g["ig"][t]).reshape(B, NH).to(dev)
        fg = torch.from_numpy(g["fg"][t]).reshape(B, NH).to(dev)
        _, h_raw = eng.cell_step(C, n, m, qkv.contiguous(), ig.contiguous(), fg.contiguous(), w0, B, 1)
        ref = torch.from_numpy(g["h"][t]).reshape(B, NH * DH)
        assert _rel(h_raw.cpu(), ref) < REL_TOL, f"step {t}"
    s = math.sqrt(DH)
    assert _rel(C.cpu() * s, torch.from_numpy(g["c_final"])) < 1e-4
    assert _rel(n.cpu() * s, torch.from_numpy(g["n_final"])) < 1e-4
    assert (m.cpu().view(B, NH, 1) - torch.from_numpy(g["m_final"])).abs().max() < 1e-5
    eng.close()


def test_cell_steps_from_nonzero_state_vs_hf_chunkwise_golden(golden_dir):
    """fused-T kernel, 48 tokens as 12 launches of T = 4 from a NON-ZERO (C, n, m), vs vectors from transformers'
    chunkwise-parallel forward started from the same state (independent implementation, different algorithm)."""
    g = np.load(os.path.join(golden_dir, "hf_mlstm_chunkwise.npz"))
    B, NH, S, DH = g["q"].shape
    cfg, sd, eng = _engine("toy", B)
    assert (cfg.num_heads, cfg.head_dim) == (NH, DH)
    dev, s, T = eng.device, math.sqrt(DH), 4
    C = (torch.from_numpy(g["c0"]) / s).to(dev)
    n = (torch.from_numpy(g["n0"]) / s).to(dev)
    m = torch.from_numpy(g["m0"]).reshape(B, NH).to(dev)
    w0 = torch.zeros(cfg.inner, device=dev)
    q, k, v = (torch.from_numpy(g[x]) for x in ("q", "k", "v"))          # [B,NH,S,DH]
    for t0 in range(0, S, T):
        rows = [torch.stack([x[:, :, t0 + t].reshape(B, NH * DH) for x in (q, k, v)], dim=1) for t in range(T)]
        qkv = torch.stack(rows, dim=1).reshape(B * T, 3, NH * DH).to(dev)            # row = b*T + t
        ig = torch.from_numpy(g["ig"][:, :, t0:t0 + T]).permute(0, 2, 1).reshape(B * T, NH).to(dev)
        fg = torch.from_numpy(g["fg"][:, :, t0:t0 + T]).permute(0, 2, 1).reshape(B * T, NH).to(dev)
        _, h_raw = eng.cell_step(C, n, m, qkv.contiguous(), ig.contiguous(), fg.contiguous(), w0, B, T)
        ref = torch.from_numpy(g["h"][:, :, t0:t0 + T]).permute(0, 2, 1, 3).reshape(B * T, NH * DH)
        assert _rel(h_raw.cpu(), ref) < REL_TOL, f"tokens {t0}..{t0 + T - 1}"
    assert _rel(C.cpu() * s, torch.from_numpy(g["c_final"])) < 1e-4
    assert _rel(n.cpu() * s, torch.from_numpy(g["n_final"])) < 1e-4
    assert (m.cpu().view(B, NH, 1) - torch.from_numpy(g["m_final"])).abs().max() < 1e-5
    eng.close()


@pytest.mark.parametrize("name,B,T,rs,cols", [("toy", 3, 1, 0, 0), ("toy", 3, 3, 0, 0), ("toy", 2, 4, 2, 16),
                                              ("toy128", 2, 3, 4, 32), ("16M", 2, 3, 0, 0), ("16M", 1, 1, 8, 64),
                                              ("48M", 2, 3, 0, 0), ("206M", 1, 3, 0, 0), ("206M", 1, 2, 5, 128)])
def test_cell_step_vs_oracle(name, B, T, rs, cols):
    """fused-T kernel == T sequential oracle steps (+ GroupNorm), for every tiling."""
    from oracle import xlstm_oracle as O
    cfg, sd, eng = _engine(name, B, num_blocks=1)
    NH, DH, inner = cfg.num_heads, cfg.head_dim, cfg.inner
    g = torch.Generator().manual_seed(42)
    C0 = torch.randn(B, NH, DH, DH, generator=g) * 0.1
    n0 = torch.randn(B, NH, DH, generator=g) * 0.1
    m0 = torch.randn(B, NH, generator=g)
    qkv = torch.randn(B * T, 3, inner, generator=g)
    ig = torch.randn(B * T, NH, generator=g) * 2
    fg = torch.randn(B * T, NH, generator=g) * 2 + 2
    w = torch.randn(inner, generator=g) * 0.1
    dev = eng.device
    C, n, m = C0.to(dev), n0.to(dev), m0.to(dev)
    h_norm, h_raw = eng.cell_step(C, n, m, qkv.to(dev), ig.to(dev), fg.to(dev), w.to(dev), B, T, rs, cols)
    torch.cuda.synchronize()
    # oracle: T sequential steps
    c, nn, mm = C0.clone(), n0.clone().unsqueeze(-1), m0.clone().view(B, NH, 1, 1)
    qv = qkv.view(B, T, 3, NH, DH)
    for t in range(T):
        q, k, v = (qv[:, t, j].unsqueeze(2) for j in range(3))              # [B,NH,1,DH]
        h, (c, nn, mm) = O.recurrent_step_stabilized_simple(
            c, nn, mm, q, k, v, ig.view(B, T, NH)[:, t].view(B, NH, 1, 1), fg.view(B, T, NH)[:, t].view(B, NH, 1, 1))
        hn = O.multihead_layer_norm(h, w).transpose(1, 2).reshape(B, inner)
        got_raw = h_raw.view(B, T, inner)[:, t].cpu()
        got = h_norm.view(B, T, inner)[:, t].cpu()
        assert _rel(got_raw, h.transpose(1, 2).reshape(B, inner)) < REL_TOL, f"h_raw t={t}"
        assert _rel(got, hn) < REL_TOL, f"h_norm t={t}"
    assert _rel(C.cpu(), c) < 1e-5
    assert _rel(n.cpu(), nn.squeeze(-1)) < 1e-5
    assert (m.cpu() - mm.view(B, NH)).abs().max() < 1e-5
    eng.close()


@pytest.mark.parametrize("name,B,T", [("48M", 5, 3), ("16M", 3, 1), ("206M", 2, 4), ("110M", 2, 3)])
def test_state_impls_agree(name, B, T):
    """impl 2 (persistent ring), impl 1 (one-shot TMA ring) and impl 0 (plain loads) run the same per-element
    arithmetic: C, n, m bit-identical; h differs only by the order of the row-chunk partial sums."""
    cfg, sd, eng = _engine(name, B, num_blocks=1)
    NH, DH, inner = cfg.num_heads, cfg.head_dim, cfg.inner
    g = torch.Generator().manual_seed(7)
    C0 = torch.randn(B, NH, DH, DH, generator=g) * 0.1
    n0 = torch.randn(B, NH, DH, generator=g) * 0.1
    m0 = torch.randn(B, NH, generator=g)
    qkv = (torch.randn(B * T, 3, inner, generator=g)).cuda()
    ig = (torch.randn(B * T, NH, generator=g) * 2).cuda()
    fg = (torch.randn(B * T, NH, generator=g) * 2 + 2).cuda()
    w = (torch.randn(inner, generator=g) * 0.1).cuda()
    res = {}
    variants = [(0, {}), (1, {}), (2, {}), (2, {"state_stages": 3, "state_ctas_per_sm": 2})]
    for k, (impl, opts) in enumerate(variants):
        eng.set_option("state_impl", impl)
        for o in ("state_stages", "state_ctas_per_sm"):
            eng.set_option(o, opts.get(o, 0))
        C, n, m = C0.cuda(), n0.cuda(), m0.cuda()
        for _ in range(2):                                   # two steps: the second consumes the updated state
            h_norm, h_raw = eng.cell_step(C, n, m, qkv, ig, fg, w, B, T)
        torch.cuda.synchronize()
        res[k] = (C.cpu(), n.cpu(), m.cpu(), h_norm.cpu(), h_raw.cpu())
    for k in range(1, len(variants)):
        assert torch.equal(res[k][0], res[0][0]), f"C differs: variant {k}"
        assert torch.equal(res[k][1], res[0][1]) and torch.equal(res[k][2], res[0][2])
        assert _rel(res[k][3], res[0][3]) < 1e-5 and _rel(res[k][4], res[0][4]) < 1e-5
    eng.close()


# ------------------------------------------------------------------------------------------------------------
# unit: Linear
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K", [(1, 64, 64), (3, 2192, 128), (192, 3072, 768), (100, 768, 1536), (64, 512, 256)])
def test_linear_vs_torch(M, N, K):
    cfg, sd, eng = _engine("toy", 1)
    g = torch.Generator().manual_seed(M * 7 + N)
    A = torch.randn(M, K, generator=g)
    W = (torch.randn(N, K, generator=g) * 0.05).to(torch.bfloat16)
    bias = torch.randn(N, generator=g)
    res = torch.randn(M, N, generator=g)
    ref = (A.double() @ W.double().t() + bias.double() + res.double()).float()
    out = eng.linear(A.cuda(), W.cuda(), bias.cuda(), res.cuda())
    assert _rel(out.cpu(), ref) < 1e-5
    out2 = eng.linear(A.cuda(), W.cuda())
    assert _rel(out2.cpu(), (A.double() @ W.double().t()).float()) < 1e-5
    eng.close()


# ------------------------------------------------------------------------------------------------------------
# integration: encoder, both modes
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,B,mode", [("toy", 4, L.XL_MODE_PER_TOKEN), ("toy", 4, L.XL_MODE_FUSED),
                                         ("toy128", 3, L.XL_MODE_FUSED), ("16M", 2, L.XL_MODE_FUSED),
                                         ("16M", 1, L.XL_MODE_PER_TOKEN)])
def test_encoder_step_vs_oracle(name, B, mode):
    from lram_b200.decision_xlstm import FusedXLSTMEncoder
    from oracle import xlstm_oracle as O
    cfg, sd, eng = _engine(name, B)
    enc = FusedXLSTMEncoder(eng, mode=mode)
    ora = O.OracleEncoder(cfg, sd)
    g = torch.Generator().manual_seed(9)
    pkv_o, pkv = None, None
    for step in range(3):
        x = torch.randn(B, 3, cfg.d, generator=g)
        out = enc(inputs_embeds=x.cuda(), past_key_values=pkv, use_cache=True)
        pkv = out["past_key_values"]
        ref, pkv_o = ora.forward_cached(x, pkv_o)
        assert _rel(out["last_hidden_state"].cpu(), ref) < REL_TOL, f"step {step}"
    # state export in the reference's past_key_values format
    exp = pkv.to_past_key_values()
    for i in range(cfg.num_blocks):
        c, n, m = pkv_o[f"block_{i}"]["mlstm_state"]
        ce, ne, me = exp[f"block_{i}"]["mlstm_state"]
        assert _rel(ce.cpu(), c) < REL_TOL and _rel(ne.cpu(), n) < REL_TOL
        assert (me.cpu() - m).abs().max() < 1e-4
        assert _rel(exp[f"block_{i}"]["conv_state"][0].cpu(), pkv_o[f"block_{i}"]["conv_state"][0]) < 1e-5
    # import: continue from the ORACLE's state and match again
    x = torch.randn(B, 3, cfg.d, generator=g)
    out = enc(inputs_embeds=x.cuda(), past_key_values=pkv_o, use_cache=True)
    ref, _ = ora.forward_cached(x, pkv_o)
    assert _rel(out["last_hidden_state"].cpu(), ref) < REL_TOL
    eng.close()


# ------------------------------------------------------------------------------------------------------------
# integration: whole policy step vs committed golden vectors + oracle
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["toy", "toy128"])
@pytest.mark.parametrize("mode", [L.XL_MODE_PER_TOKEN, L.XL_MODE_FUSED])
def test_policy_step_vs_golden(golden_dir, name, mode):
    g = np.load(os.path.join(golden_dir, "oracle_toy.npz"))
    states, rtg = g[f"{name}_states"], g[f"{name}_rtg"]
    steps, B = rtg.shape
    cfg, sd, eng = _engine(name, B)
    cache = eng.new_state(B)
    for t in range(steps):
        out = eng.policy_step(cache, torch.from_numpy(states[t]).cuda(), torch.from_numpy(rtg[t]).cuda(), mode=mode,
                              want_hidden=True, want_logits=True)
        torch.cuda.synchronize()
        assert np.array_equal(out["action_tokens"].cpu().numpy().astype(np.int64), g[f"{name}_tokens"][t]), f"t={t}"
        assert np.array_equal(out["action_preds"].cpu().numpy(), g[f"{name}_actions"][t])
        assert _rel(out["last_hidden_state"].cpu(), torch.from_numpy(g[f"{name}_hidden"][t])) < REL_TOL
    last = cfg.num_blocks - 1
    assert _rel(cache.c_logical(last).cpu(), torch.from_numpy(g[f"{name}_C_last"])) < REL_TOL
    assert _rel(cache.view(last, L.XL_STATE_CONV).cpu(), torch.from_numpy(g[f"{name}_conv_last"])) < 1e-5
    eng.close()


@pytest.mark.parametrize("name,B,steps", [("16M", 4, 4), ("48M", 3, 3)])
def test_policy_step_real_sizes_vs_oracle(name, B, steps):
    from oracle import xlstm_oracle as O
    cfg, sd, eng = _engine(name, B)
    ora = O.OraclePolicy(cfg, sd)
    states, rtg, _ = make_stream(cfg, range(B), steps, domains="mixed")
    cache, pkv = eng.new_state(B), None
    for t in range(steps):
        out = eng.policy_step(cache, torch.from_numpy(states[t]).cuda(), torch.from_numpy(rtg[t]).cuda(),
                              mode=L.XL_MODE_FUSED, want_hidden=True, want_logits=True)
        ref = ora.step(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), past_key_values=pkv)
        pkv = ref["past_key_values"]
        tok = out["action_tokens"].cpu().long()
        margins = _margin_ok(ref["action_logits"], tok, ref["action_tokens"])
        assert not margins, f"token mismatches at t={t}, oracle top-2 relative margins {margins}"
        assert _rel(out["last_hidden_state"].cpu(), ref["last_hidden_state"]) < REL_TOL
        assert torch.equal(out["action_preds"].cpu(), ref["action_preds"])
        assert _rel(out["action_logits"].cpu().view_as(ref["action_logits"]), ref["action_logits"]) < REL_TOL
    eng.close()


def test_discrete_branch_vs_oracle():
    from oracle import xlstm_oracle as O
    cfg, sd, eng = _engine("toy128", 5)
    ora = O.OraclePolicy(cfg, sd)
    states, rtg, _ = make_stream(cfg, range(5), 3, domains="mixed")
    cache, pkv = eng.new_state(5), None
    for t in range(3):
        out = eng.policy_step(cache, torch.from_numpy(states[t]).cuda(), torch.from_numpy(rtg[t]).cuda(),
                              flags=L.XL_FLAG_DISCRETE, want_logits=True)
        ref = ora.step(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), past_key_values=pkv, discrete=True)
        pkv = ref["past_key_values"]
        assert torch.equal(out["action_tokens"].cpu().long()[:, :1], ref["action_tokens"])
        assert _rel(out["action_logits"].cpu(), ref["action_logits"].view(5, -1)) < REL_TOL
    eng.close()


def test_fused_equals_per_token_and_graph_replay():
    """Properties that need no oracle: fused == per-token stepping; CUDA-graph replay == eager launches."""
    cfg, sd, eng = _engine("16M", 8)
    states, rtg, _ = make_stream(cfg, range(8), 6, domains="mixed")
    res = {}
    for tag, mode, flags in (("tok", L.XL_MODE_PER_TOKEN, 0), ("fused", L.XL_MODE_FUSED, 0),
                             ("graph", L.XL_MODE_FUSED, L.XL_FLAG_GRAPH)):
        cache = eng.new_state(8)
        s_dev = torch.empty(8, cfg.state_dim, device="cuda")
        r_dev = torch.empty(8, device="cuda")
        out = None
        toks, hids = [], []
        for t in range(6):
            s_dev.copy_(torch.from_numpy(states[t]))
            r_dev.copy_(torch.from_numpy(rtg[t]))
            out = eng.policy_step(cache, s_dev, r_dev, mode=mode, flags=flags, want_hidden=True, out=out)
            torch.cuda.synchronize()
            toks.append(out["action_tokens"].cpu().clone())
            hids.append(out["last_hidden_state"].cpu().clone())
        res[tag] = (torch.stack(toks), torch.stack(hids))
    assert torch.equal(res["tok"][0], res["fused"][0])
    assert _rel(res["fused"][1], res["tok"][1]) < 1e-4
    assert torch.equal(res["graph"][0], res["fused"][0])
    assert torch.equal(res["graph"][1], res["fused"][1])          # same kernels, same order: bit identical
    eng.close()


# ------------------------------------------------------------------------------------------------------------
# context prefill (SURVEY §8 a11 / BASELINE configs[3])
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,B,S", [("toy128", 3, 50), ("toy128", 2, 7), ("16M", 2, 36), ("toy", 2, 21),
                                      ("48M", 1, 24)])
def test_prefill_vs_oracle_steps(name, B, S):
    """xl_prefill over S tokens == S recurrent oracle steps: hidden states of every token and the state left."""
    from lram_b200.decision_xlstm import FusedXLSTMEncoder
    from oracle import xlstm_oracle as O
    cfg, sd, eng = _engine(name, B)
    ora = O.OracleEncoder(cfg, sd)
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, S, cfg.d, generator=g)
    # start from a non-trivial state: 2 tokens through the step path on both sides
    x0 = torch.randn(B, 2, cfg.d, generator=g)
    enc = FusedXLSTMEncoder(eng, mode=L.XL_MODE_FUSED)
    out0 = enc(inputs_embeds=x0.cuda(), past_key_values=None, use_cache=True)
    cache = out0["past_key_values"]
    _, pkv_o = ora.forward_cached(x0, None)
    out = enc(inputs_embeds=x.cuda(), past_key_values=cache, use_cache=True)       # S > 4 -> prefill path
    refs = []
    for t in range(S):
        r, pkv_o = ora.forward_cached(x[:, t:t + 1], pkv_o)
        refs.append(r)
    ref = torch.cat(refs, dim=1)
    assert _rel(out["last_hidden_state"].cpu(), ref) < REL_TOL
    exp = cache.to_past_key_values()
    for i in range(cfg.num_blocks):
        c, n, m = pkv_o[f"block_{i}"]["mlstm_state"]
        ce, ne, me = exp[f"block_{i}"]["mlstm_state"]
        assert _rel(ce.cpu(), c) < REL_TOL and _rel(ne.cpu(), n) < REL_TOL, f"block {i}"
        assert (me.cpu() - m).abs().max() < 1e-4
        assert _rel(exp[f"block_{i}"]["conv_state"][0].cpu(), pkv_o[f"block_{i}"]["conv_state"][0]) < 1e-5
    # and the rollout continues from the prefilled state exactly like from the stepped one
    x1 = torch.randn(B, 3, cfg.d, generator=g)
    o1 = enc(inputs_embeds=x1.cuda(), past_key_values=cache, use_cache=True)
    r1, _ = ora.forward_cached(x1, pkv_o)
    assert _rel(o1["last_hidden_state"].cpu(), r1) < REL_TOL
    eng.close()


@pytest.mark.parametrize("name,B,S", [("16M", 2, 304), ("110M", 1, 176), ("206M", 1, 144)])
def test_prefill_cells_agree_and_match_oracle_steps(name, B, S):
    """The three sequence cells of the context prefill -- chunkwise tcgen05 (default, xl_prefill_tc.cu: 128-token chunks,
    S here spans a ragged last chunk), chunkwise mma.sync (16-token chunks) and the fp32 token-order cell -- must leave
    the same hidden states and recurrent state, and that state must be what S sequential oracle steps leave."""
    from oracle import xlstm_oracle as O
    cfg, sd, eng = _engine(name, B)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, S, cfg.d, generator=g)
    res = {}
    for cell in (2, 1, 0):
        eng.set_option("prefill_cell", cell)
        cache = eng.new_state(B)
        eng.launch_count()
        hs = eng.prefill(cache, x.cuda())
        torch.cuda.synchronize()
        res[cell] = (hs.cpu(), cache.to_past_key_values(), eng.launch_count())
    eng.set_option("prefill_cell", 2)
    assert res[2][2] > res[1][2]          # the tcgen05 cell is several launches per block: proof that it ran
    for cell in (1, 0):
        assert _rel(res[cell][0], res[2][0]) < 1e-4, cell
        for i in range(cfg.num_blocks):
            for a, b in zip(res[cell][1][f"block_{i}"]["mlstm_state"], res[2][1][f"block_{i}"]["mlstm_state"]):
                assert _rel(a.cpu(), b.cpu()) < 1e-4 or (a.cpu() - b.cpu()).abs().max() < 1e-5, (cell, i)
    ora = O.OracleEncoder(cfg, sd)
    pkv, refs = None, []
    for t in range(S):
        r, pkv = ora.forward_cached(x[:, t:t + 1], pkv)
        refs.append(r)
    assert _rel(res[2][0], torch.cat(refs, dim=1)) < REL_TOL
    for i in range(cfg.num_blocks):
        c, n, m = pkv[f"block_{i}"]["mlstm_state"]
        ce, ne, me = res[2][1][f"block_{i}"]["mlstm_state"]
        assert _rel(ce.cpu(), c) < REL_TOL and _rel(ne.cpu(), n) < REL_TOL, f"block {i}"
        assert (me.cpu() - m).abs().max() < 1e-4
    eng.close()


@pytest.mark.parametrize("name,B,S", [("16M", 2, 301), ("48M", 3, 75), ("206M", 1, 130), ("toy128", 2, 37)])
def test_prefill_conv_packed_fp32_equals_scalar(name, B, S):
    """xl_set_option("prefill_conv"): the sequence conv/qkv/gates kernel on packed fp32 pairs (FFMA2, 1) keeps every FMA
    chain of the scalar kernel (0), so hidden states and the state left are BIT-identical; 2 (the default: + SFU SiLU)
    differs by the ~2 ulp of ex2.approx / rcp.approx. xl_set_option("prefill_prep"): the single-read chunk preparation
    (shared-memory tile, default = 1) writes the same operand planes as the three-pass kernel (0), bit for bit.
    S is ragged against the 2-token groups, the 16-token runs and the 128-token chunks; the first call starts from a
    carried conv window and a non-zero state."""
    cfg, sd, eng = _engine(name, B)
    g = torch.Generator().manual_seed(23)
    x0 = torch.randn(B, 9, cfg.d, generator=g)
    x = torch.randn(B, S, cfg.d, generator=g)
    res = {}
    try:
        for tag, conv, prep in (("base", 0, 0), ("conv1", 1, 0), ("prep1", 0, 1), ("fast", 2, 1)):
            eng.set_option("prefill_conv", conv)
            eng.set_option("prefill_prep", prep)
            cache = eng.new_state(B)
            eng.prefill(cache, x0.cuda())
            hs = eng.prefill(cache, x.cuda())
            torch.cuda.synchronize()
            res[tag] = (hs.cpu(), cache.to_past_key_values())
    finally:
        eng.set_option("prefill_conv", 2)       # process-wide switches: restore the defaults
        eng.set_option("prefill_prep", 1)
    for tag in ("conv1", "prep1"):
        assert torch.equal(res[tag][0], res["base"][0]), tag
    assert _rel(res["fast"][0], res["base"][0]) < 1e-4
    for i in range(cfg.num_blocks):
        base = res["base"][1][f"block_{i}"]
        for tag in ("conv1", "prep1"):
            blk = res[tag][1][f"block_{i}"]
            for a, b in zip(base["mlstm_state"], blk["mlstm_state"]):
                assert torch.equal(a.cpu(), b.cpu()), (tag, i)
            assert torch.equal(base["conv_state"][0].cpu(), blk["conv_state"][0].cpu()), (tag, i)
        for a, c in zip(base["mlstm_state"], res["fast"][1][f"block_{i}"]["mlstm_state"]):
            assert _rel(c.cpu(), a.cpu()) < 1e-4 or (c.cpu() - a.cpu()).abs().max() < 1e-5, i
    eng.close()


@pytest.mark.parametrize("name,B,S", [("206M", 1, 300), ("48M", 2, 200), ("16M", 8, 130)])
def test_prefill_tc_side_stream_overlap_equals_sequential(name, B, S):
    """xl_set_option("prefill_tc_overlap"): with few envs the S = QK^T GEMM (grid capped at the SMs the chunk scan leaves
    free), the P~ kernel and the n scan run on a side stream beside the chunk update + scan and join before the numerator
    GEMM. Same kernels, same tiles: bit-identical to the single-stream order (16M x 8 envs: 128 scan CTAs, no overlap)."""
    cfg, sd, eng = _engine(name, B)
    g = torch.Generator().manual_seed(29)
    x = torch.randn(B, S, cfg.d, generator=g)
    res = {}
    try:
        for ovl in (0, 1, 0, 1):          # twice: the side stream's workspace reuse across calls and blocks is ordered
            eng.set_option("prefill_tc_overlap", ovl)
            cache = eng.new_state(B)
            hs = eng.prefill(cache, x.cuda())
            hs2 = eng.prefill(cache, x.flip(1).contiguous().cuda())
            torch.cuda.synchronize()
            out = (hs.cpu(), hs2.cpu(), cache.to_past_key_values())
            if ovl in res:
                assert torch.equal(out[0], res[ovl][0]) and torch.equal(out[1], res[ovl][1])
            res[ovl] = out
    finally:
        eng.set_option("prefill_tc_overlap", 1)
    assert torch.equal(res[1][0], res[0][0]) and torch.equal(res[1][1], res[0][1])
    for i in range(cfg.num_blocks):
        for a, b in zip(res[0][2][f"block_{i}"]["mlstm_state"], res[1][2][f"block_{i}"]["mlstm_state"]):
            assert torch.equal(a.cpu(), b.cpu()), i
    eng.close()


@pytest.mark.parametrize("name,B,S", [("206M", 1, 300), ("16M", 3, 200)])
def test_prefill_scan_epilogue_split_is_bit_identical(name, B, S):
    """xl_set_option("prefill_scan_split"): the chunk update + scan kernel with 16 epilogue warps (4 per TMEM lane quarter,
    32 columns of the C^T tile per thread) instead of 8 (2 per quarter, 64 columns): same arithmetic per element."""
    cfg, sd, eng = _engine(name, B)
    g = torch.Generator().manual_seed(31)
    x = torch.randn(B, S, cfg.d, generator=g)
    res = {}
    try:
        for split in (2, 4):
            eng.set_option("prefill_scan_split", split)
            cache = eng.new_state(B)
            hs = eng.prefill(cache, x.cuda())
            hs2 = eng.prefill(cache, x.flip(1).contiguous().cuda())
            torch.cuda.synchronize()
            res[split] = (hs.cpu(), hs2.cpu(), cache.to_past_key_values())
    finally:
        eng.set_option("prefill_scan_split", DEFAULT_SCAN_SPLIT)
    assert torch.equal(res[4][0], res[2][0]) and torch.equal(res[4][1], res[2][1])
    for i in range(cfg.num_blocks):
        for a, b in zip(res[2][2][f"block_{i}"]["mlstm_state"], res[4][2][f"block_{i}"]["mlstm_state"]):
            assert torch.equal(a.cpu(), b.cpu()), i
    eng.close()


@pytest.mark.parametrize("Tn", [23, 100])
def test_policy_prefill_equals_stepping(Tn):
    """xl_policy_prefill(context of Tn timesteps) then a rollout == stepping through the context: same action
    tokens afterwards (needs no oracle: both sides are this library; the step path is oracle-checked above).
    Tn = 23: one ragged 64-token chunk + stepped tail; Tn = 100: 300 tokens of 3 envs = 128 + 128 + 44 through the tcgen05 cell."""
    cfg, sd, eng = _engine("16M", 3)
    Tr = 4
    states, rtg, _ = make_stream(cfg, range(3), Tn + Tr, domains="mixed")
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    stepped = eng.new_state(3)
    for t in range(Tn):
        eng.policy_step(stepped, dev(states[t]), dev(rtg[t]))
    pre = eng.new_state(3)
    eng.policy_prefill(pre, dev(states[:Tn].transpose(1, 0, 2)), dev(rtg[:Tn].T))
    for i in range(cfg.num_blocks):
        assert _rel(pre.c_logical(i).cpu(), stepped.c_logical(i).cpu()) < 1e-4, f"block {i}"
        assert (pre.view(i, L.XL_STATE_M) - stepped.view(i, L.XL_STATE_M)).abs().max().item() < 1e-4
    for t in range(Tn, Tn + Tr):
        a = eng.policy_step(stepped, dev(states[t]), dev(rtg[t]), want_hidden=True)
        b = eng.policy_step(pre, dev(states[t]), dev(rtg[t]), want_hidden=True)
        torch.cuda.synchronize()
        assert torch.equal(a["action_tokens"].cpu(), b["action_tokens"].cpu())
        assert _rel(b["last_hidden_state"].cpu(), a["last_hidden_state"].cpu()) < 1e-4
    eng.close()


def test_per_env_reset_mask():
    """reset of a subset of envs == those envs starting from past_key_values=None; others untouched."""
    cfg, sd, eng = _engine("toy128", 4)
    states, rtg, _ = make_stream(cfg, range(4), 4, domains="mixed")
    dev = lambda a: torch.from_numpy(a).cuda()
    cache = eng.new_state(4)
    for t in range(2):
        eng.policy_step(cache, dev(states[t]), dev(rtg[t]))
    eng.reset(cache, torch.tensor([0, 1, 0, 1], dtype=torch.uint8))
    out = eng.policy_step(cache, dev(states[2]), dev(rtg[2]), want_hidden=True)
    fresh = eng.new_state(4)
    out_f = eng.policy_step(fresh, dev(states[2]), dev(rtg[2]), want_hidden=True)
    cont = eng.new_state(4)
    for t in range(3):
        out_c = eng.policy_step(cont, dev(states[t]), dev(rtg[t]), want_hidden=True)
    torch.cuda.synchronize()
    h, hf, hc = (o["last_hidden_state"].cpu() for o in (out, out_f, out_c))
    assert torch.equal(h[[1, 3]], hf[[1, 3]])
    assert torch.equal(h[[0, 2]], hc[[0, 2]])
    eng.close()


def test_host_step_and_agent_predict_b1():
    """The reference-facing call chain for one env: agent.predict -> policy.forward -> library; and the host
    (pinned) step used by the rollout loop."""
    from lram_b200.decision_xlstm import DiscreteDecisionXLSTM, MultiDomainDiscreteDecisionXLSTMModel
    from oracle import xlstm_oracle as O
    cfg = preset("toy128")
    sd = make_state_dict(cfg, seed=0)
    policy = MultiDomainDiscreteDecisionXLSTMModel(cfg, sd, max_batch=1)
    agent = DiscreteDecisionXLSTM(policy)
    ora = O.OraclePolicy(cfg, sd)
    states, rtg, envs = make_stream(cfg, [0], 4, domains="metaworld")
    act_dim = int(envs.act_dims[0])
    pkv = None
    actions = torch.zeros((0, act_dim), device="cuda")
    for t in range(4):
        actions = torch.cat([actions, torch.zeros((1, act_dim), device="cuda")], dim=0)
        rewards = torch.zeros(t + 1, device="cuda")
        obs = torch.from_numpy(states[: t + 1, 0, :39]).cuda()           # raw 39-dim Meta-World obs, unpadded
        a, _ = agent.predict(policy, obs, actions, rewards, torch.from_numpy(rtg[: t + 1, 0]).cuda().reshape(1, -1),
                             torch.arange(t + 1, device="cuda").reshape(1, -1), context_len=1, env_act_dim=act_dim)
        ref = ora.step(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), past_key_values=pkv)
        pkv = ref["past_key_values"]
        assert a.shape == (act_dim,)
        assert torch.equal(a.cpu(), ref["action_preds"][0, :act_dim])
        actions[-1] = a
    # host-buffer entry point
    eng = policy.engine
    cache = eng.new_state(1)
    hs = torch.from_numpy(states[0]).pin_memory()
    hr = torch.from_numpy(rtg[0]).pin_memory()
    ht = torch.zeros(1, cfg.act_dim, dtype=torch.int32).pin_memory()
    ha = torch.zeros(1, cfg.act_dim).pin_memory()
    eng.policy_step_host(cache, hs, hr, ht, ha)
    ref0 = ora.step(torch.from_numpy(states[0]), torch.from_numpy(rtg[0]))
    assert torch.equal(ht.long(), ref0["action_tokens"])
    eng.close()


def test_long_horizon_drift_and_rollout_driver():
    """200 env steps with resets through the batched rollout driver: tokens must stay bit-exact vs the oracle."""
    from lram_b200.engine import XLSTMEngine
    from lram_b200.rollout import BatchedRollout
    from lram_b200.synth import SyntheticEnvBatch
    from oracle import xlstm_oracle as O
    cfg = preset("toy")
    sd = make_state_dict(cfg, seed=0)
    B, steps, ep_len = 4, 200, 37
    eng = XLSTMEngine(cfg, sd, max_batch=B)
    ro = BatchedRollout(eng, SyntheticEnvBatch(cfg, range(B), domains="mixed", ep_len=ep_len), use_graph=True)
    res = ro.run(steps, record=True)
    # oracle replay of the same loop
    ora = O.OraclePolicy(cfg, sd)
    envs = SyntheticEnvBatch(cfg, range(B), domains="mixed", ep_len=ep_len)
    obs, rtg, pkv = envs.reset(), envs.rtg0.copy(), None
    mism = 0
    for t in range(steps):
        o = ora.step(torch.from_numpy(obs), torch.from_numpy(rtg), past_key_values=pkv)
        pkv = o["past_key_values"]
        mism += int((o["action_tokens"].numpy() != res["tokens"][t]).sum())
        obs, rew, done = envs.step(None)
        rtg = (rtg - rew / envs.reward_scale).astype(np.float32)
        if done.any():
            rtg[done] = envs.rtg0[done]
            pkv = O.reset_state_rows(pkv, torch.from_numpy(done))
    assert mism == 0, f"{mism} token mismatches over {steps * B * cfg.act_dim}"
    assert len(res["episode_returns"][0]) == steps // ep_len
    eng.close()


# ------------------------------------------------------------------------------------------------------------
# xLSTM[a:b] stacks: sLSTM blocks (SURVEY §8 f4; xlstm_ms_mediumplus.yaml:27 slstm_at: [1])
# ------------------------------------------------------------------------------------------------------------
def _assert_states_match(cfg, exp, pkv_o, tol=REL_TOL):
    for i in range(cfg.num_blocks):
        eo, oo = exp[f"block_{i}"], pkv_o[f"block_{i}"]
        assert _rel(eo["conv_state"][0].cpu(), oo["conv_state"][0]) < 1e-5, f"block {i} conv"
        if cfg.is_slstm(i):
            se, so = eo["slstm_state"].cpu(), oo["slstm_state"]
            for part, nm in enumerate("ycnm"):
                assert _rel(se[part], so[part]) < tol, f"block {i} sLSTM {nm}"
            continue
        c, n, m = oo["mlstm_state"]
        ce, ne, me = eo["mlstm_state"]
        assert _rel(ce.cpu(), c) < tol and _rel(ne.cpu(), n) < tol, f"block {i}"
        assert (me.cpu() - m).abs().max() < 1e-4


@pytest.mark.parametrize("name,B,mode", [("toy-ms", 4, L.XL_MODE_PER_TOKEN), ("toy-ms", 4, L.XL_MODE_FUSED),
                                         ("toy128-ms", 11, L.XL_MODE_FUSED), ("48M-ms", 2, L.XL_MODE_FUSED)])
def test_slstm_encoder_step_vs_oracle(name, B, mode):
    from lram_b200.decision_xlstm import FusedXLSTMEncoder
    from oracle import xlstm_oracle as O
    cfg, sd, eng = _engine(name, B)
    enc = FusedXLSTMEncoder(eng, mode=mode)
    ora = O.OracleEncoder(cfg, sd)
    g = torch.Generator().manual_seed(19)
    pkv_o, pkv = None, None
    for step in range(4):
        x = torch.randn(B, 3, cfg.d, generator=g)
        out = enc(inputs_embeds=x.cuda(), past_key_values=pkv, use_cache=True)
        pkv = out["past_key_values"]
        ref, pkv_o = ora.forward_cached(x, pkv_o)
        assert _rel(out["last_hidden_state"].cpu(), ref) < REL_TOL, f"step {step}"
    _assert_states_match(cfg, pkv.to_past_key_values(), pkv_o)
    # import the ORACLE's state (reference past_key_values format incl. "slstm_state") and continue
    x = torch.randn(B, 3, cfg.d, generator=g)
    out = enc(inputs_embeds=x.cuda(), past_key_values=pkv_o, use_cache=True)
    ref, _ = ora.forward_cached(x, pkv_o)
    assert _rel(out["last_hidden_state"].cpu(), ref) < REL_TOL
    eng.close()


@pytest.mark.parametrize("name,B,steps", [("toy128-ms", 6, 5), ("48M-ms", 3, 3)])
def test_slstm_policy_step_tokens_bit_exact(name, B, steps):
    from oracle import xlstm_oracle as O
    cfg, sd, eng = _engine(name, B)
    ora = O.OraclePolicy(cfg, sd)
    states, rtg, _ = make_stream(cfg, range(B), steps, domains="mixed")
    cache, cache_g, pkv = eng.new_state(B), eng.new_state(B), None
    for t in range(steps):
        s_t, r_t = torch.from_numpy(states[t]).cuda(), torch.from_numpy(rtg[t]).cuda()
        out = eng.policy_step(cache, s_t, r_t, mode=L.XL_MODE_FUSED, want_hidden=True, want_logits=True)
        ref = ora.step(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), past_key_values=pkv)
        pkv = ref["past_key_values"]
        tok = out["action_tokens"].cpu().long()
        margins = _margin_ok(ref["action_logits"], tok, ref["action_tokens"])
        assert not margins, f"token mismatches at t={t}, oracle top-2 relative margins {margins}"
        assert _rel(out["last_hidden_state"].cpu(), ref["last_hidden_state"]) < REL_TOL
        assert torch.equal(out["action_preds"].cpu(), ref["action_preds"])
        # CUDA-graph replay of the same step on a second cache: identical bits
        out_g = eng.policy_step(cache_g, s_t, r_t, mode=L.XL_MODE_FUSED, flags=L.XL_FLAG_GRAPH, want_hidden=True)
        torch.cuda.synchronize()
        assert torch.equal(out_g["action_tokens"].cpu(), out["action_tokens"].cpu())
        assert torch.equal(out_g["last_hidden_state"].cpu(), out["last_hidden_state"].cpu())
    eng.close()


def test_slstm_prefill_and_reset():
    """sLSTM stacks through the other entry points: context prefill == stepping, per-env reset == fresh state."""
    from lram_b200.decision_xlstm import FusedXLSTMEncoder
    from oracle import xlstm_oracle as O
    cfg, sd, eng = _engine("toy128-ms", 4)
    B, S = 4, 30
    ora = O.OracleEncoder(cfg, sd)
    g = torch.Generator().manual_seed(23)
    x = torch.randn(B, S, cfg.d, generator=g)
    enc = FusedXLSTMEncoder(eng, mode=L.XL_MODE_FUSED)
    out = enc(inputs_embeds=x.cuda(), past_key_values=None, use_cache=True)          # S > 4 -> prefill path
    refs, pkv_o = [], None
    for t in range(S):
        r, pkv_o = ora.forward_cached(x[:, t:t + 1], pkv_o)
        refs.append(r)
    assert _rel(out["last_hidden_state"].cpu(), torch.cat(refs, dim=1)) < REL_TOL
    cache = out["past_key_values"]
    _assert_states_match(cfg, cache.to_past_key_values(), pkv_o)
    # per-env reset
    states, rtg, _ = make_stream(cfg, range(B), 3, domains="mixed")
    dev = lambda a: torch.from_numpy(a).cuda()
    c1 = eng.new_state(B)
    for t in range(2):
        eng.policy_step(c1, dev(states[t]), dev(rtg[t]))
    eng.reset(c1, torch.tensor([1, 0, 0, 1], dtype=torch.uint8))
    o1 = eng.policy_step(c1, dev(states[2]), dev(rtg[2]), want_hidden=True)
    of = eng.policy_step(eng.new_state(B), dev(states[2]), dev(rtg[2]), want_hidden=True)
    torch.cuda.synchronize()
    assert torch.equal(o1["last_hidden_state"].cpu()[[0, 3]], of["last_hidden_state"].cpu()[[0, 3]])
    eng.close()


def test_l2_warm_option_is_value_neutral():
    """xl_set_option("l2_prefetch_mb"): the side-stream L2 warm-up only reads; results are bit-identical."""
    cfg, sd, eng = _engine("16M", 3)
    states, rtg, _ = make_stream(cfg, range(3), 3, domains="mixed")
    dev = lambda a: torch.from_numpy(a).cuda()
    ca, cb = eng.new_state(3), eng.new_state(3)
    for t in range(3):
        eng.set_option("l2_prefetch_mb", 0)
        a = eng.policy_step(ca, dev(states[t]), dev(rtg[t]), flags=L.XL_FLAG_GRAPH, want_hidden=True)
        a = {k: v.clone() for k, v in a.items()}
        eng.set_option("l2_prefetch_mb", 8)
        b = eng.policy_step(cb, dev(states[t]), dev(rtg[t]), flags=L.XL_FLAG_GRAPH, want_hidden=True)
        torch.cuda.synchronize()
        assert torch.equal(a["action_tokens"].cpu(), b["action_tokens"].cpu())
        assert torch.equal(a["last_hidden_state"].cpu(), b["last_hidden_state"].cpu())
    eng.close()


@pytest.mark.parametrize("name,B,mode", [("48M", 16, L.XL_MODE_FUSED), ("16M", 64, L.XL_MODE_FUSED),
                                         ("toy128", 5, L.XL_MODE_FUSED), ("16M", 9, L.XL_MODE_PER_TOKEN)])
def test_conv_impl_token_parallel_is_bit_identical(name, B, mode):
    """xl_set_option("conv_impl", 1): one thread per (4-channel block, token) instead of per block; 2: the per-block kernel
    on packed fp32 pairs (FFMA2) with the gate weights loaded before the dependency wait and a butterfly reduction. Same
    arithmetic and the same summation order of the gate partials, so hidden states, tokens and the conv window are
    bit-identical."""
    cfg, sd, eng = _engine(name, B)
    states, rtg, _ = make_stream(cfg, range(B), 4, domains="mixed")
    res = {}
    for impl in (0, 1, 2):
        eng.set_option("conv_impl", impl)
        cache = eng.new_state(B)
        toks, hids = [], []
        for t in range(4):
            out = eng.policy_step(cache, torch.from_numpy(states[t]).cuda(), torch.from_numpy(rtg[t]).cuda(), mode=mode,
                                  want_hidden=True)
            toks.append(out["action_tokens"].cpu().clone())
            hids.append(out["last_hidden_state"].cpu().clone())
        res[impl] = (torch.stack(toks), torch.stack(hids),
                     [cache.view(i, L.XL_STATE_CONV).cpu().clone() for i in range(cfg.num_blocks)],
                     cache.view(cfg.num_blocks - 1, L.XL_STATE_C).cpu().clone())
    for impl in (1, 2):
        assert torch.equal(res[impl][0], res[0][0]), impl
        assert torch.equal(res[impl][1], res[0][1]), impl
        for a, b in zip(res[impl][2], res[0][2]):
            assert torch.equal(a, b), impl
        assert torch.equal(res[impl][3], res[0][3]), impl
    eng.close()


# ------------------------------------------------------------------------------------------------------------
# every BASELINE.json config at its REAL batch size, against the oracle on a row subsample
# ------------------------------------------------------------------------------------------------------------
def _subsample_rows(B, n=8):
    return sorted({int(round(i * (B - 1) / (n - 1))) for i in range(n)}) if B > n else list(range(B))


@pytest.mark.parametrize("name,B,discrete,domains,steps", [
    ("16M", 1, False, "dmcontrol", 4),       # configs[0]: 16M, one env, DMControl-like stream
    ("48M", 64, False, "metaworld", 3),      # configs[1]: the headline bench workload
    ("206M", 128, False, "mixed", 3),        # configs[2]: one GPU's shard (128 envs) of the 1024-env job
    ("110M", 256, True, "mixed", 3),         # configs[4]: Atari-style discrete head, 256 envs
])
def test_baseline_config_real_batch_vs_oracle_rows(name, B, discrete, domains, steps):
    """The bench path itself (fused 3-token step replayed from a CUDA graph, real batch => real tilings, split-K plans
    and L2 warm-up choices) for >= 3 env steps; batch rows are independent, so the fp32 oracle runs on <= 8 rows.
    Tokens / argmax actions bit-exact, hidden states and logits within REL_TOL, recurrent state of the sampled envs too."""
    from oracle import xlstm_oracle as O
    cfg, sd, eng = _engine(name, B, seed=3)
    rows = _subsample_rows(B)
    ora = O.OraclePolicy(cfg, sd)
    states, rtg, _ = make_stream(cfg, range(B), steps, domains=domains, seed=777)
    if discrete:      # Atari observations are frames; their embeddings enter as state tokens (SURVEY §8d config 5)
        gen = torch.Generator().manual_seed(5)
        emb = torch.randn(steps, B, cfg.d, generator=gen).clamp_min(0)           # post-ReLU like embed_image output
    flags = L.XL_FLAG_GRAPH | (L.XL_FLAG_DISCRETE if discrete else 0)
    cache, pkv, out = eng.new_state(B), None, None
    s_dev = torch.empty(B, cfg.d if discrete else cfg.state_dim, device="cuda")
    r_dev = torch.empty(B, device="cuda")
    for t in range(steps):
        s_cpu = emb[t] if discrete else torch.from_numpy(states[t])
        s_dev.copy_(s_cpu)
        r_dev.copy_(torch.from_numpy(rtg[t]))
        out = eng.policy_step(cache, s_dev, r_dev, mode=L.XL_MODE_FUSED, flags=flags, want_hidden=True,
                              want_logits=True, out=out, state_embeds=discrete)
        torch.cuda.synchronize()
        ref = ora.step(s_cpu[rows], torch.from_numpy(rtg[t][rows]), past_key_values=pkv, discrete=discrete,
                       state_embeds=discrete)
        pkv = ref["past_key_values"]
        tok = out["action_tokens"].cpu().long()[rows]
        if discrete:
            tok = tok[:, :1]
        lg_ref = ref["action_logits"].reshape(len(rows), -1, cfg.num_actions)
        margins = _margin_ok(lg_ref[..., :cfg.discrete_actions] if discrete else lg_ref,
                             tok.view(len(rows), -1), ref["action_tokens"].view(len(rows), -1))
        assert not margins, f"{name} x {B}: token mismatches at t={t}, oracle top-2 relative margins {margins}"
        assert _rel(out["last_hidden_state"].cpu()[rows], ref["last_hidden_state"]) < REL_TOL
        assert _rel(out["action_logits"].cpu()[rows].reshape(len(rows), -1),
                    ref["action_logits"].reshape(len(rows), -1)) < REL_TOL
        if not discrete:
            assert torch.equal(out["action_preds"].cpu()[rows], ref["action_preds"])
    for bi in (0, cfg.num_blocks - 1):
        c_ref, n_ref, m_ref = pkv[f"block_{bi}"]["mlstm_state"]
        idx = torch.tensor(rows, device="cuda")
        c_gpu = torch.index_select(cache.view(bi, L.XL_STATE_C), 0, idx)
        from lram_b200.engine import c_from_slab
        assert _rel(c_from_slab(c_gpu).cpu(), c_ref) < REL_TOL
        assert _rel(cache.view(bi, L.XL_STATE_N)[rows].cpu(), n_ref.squeeze(-1)) < REL_TOL
        assert _rel(cache.view(bi, L.XL_STATE_M)[rows].cpu(), m_ref.view(len(rows), -1)) < REL_TOL
    eng.close()


def test_fp32_checkpoint_weights_error_bound(capsys):
    """A real LRAM checkpoint holds fp32 weights; the engine rounds the four GEMM matrix families to bf16
    (north_star: "bf16 weights, fp32 state"). Against the fp32 oracle on the UNROUNDED weights this measures what that
    rounding costs over 12 blocks and 6 env steps: hidden-state error and argmax-token agreement. The bound asserted is
    loose (bf16 has 8 mantissa bits: ~4e-3 per weight, averaging down over K); INTEGRATION.md quotes the measured value."""
    from lram_b200.engine import XLSTMEngine
    from oracle import xlstm_oracle as O
    B, steps = 16, 6
    cfg = preset("48M")
    sd32 = make_state_dict(cfg, seed=9, round_bf16=False)
    eng = XLSTMEngine(cfg, sd32, max_batch=B)
    ora = O.OraclePolicy(cfg, sd32)
    states, rtg, _ = make_stream(cfg, range(B), steps, domains="mixed", seed=99)
    cache, pkv = eng.new_state(B), None
    worst_h, agree, total, flipped_margin = 0.0, 0, 0, []
    for t in range(steps):
        out = eng.policy_step(cache, torch.from_numpy(states[t]).cuda(), torch.from_numpy(rtg[t]).cuda(),
                              want_hidden=True, want_logits=True)
        ref = ora.step(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), past_key_values=pkv)
        pkv = ref["past_key_values"]
        worst_h = max(worst_h, _rel(out["last_hidden_state"].cpu(), ref["last_hidden_state"]))
        tok = out["action_tokens"].cpu().long()
        agree += int((tok == ref["action_tokens"]).sum())
        total += tok.numel()
        flipped_margin += _margin_ok(ref["action_logits"], tok, ref["action_tokens"])
    with capsys.disabled():
        print(f"\n[fp32-checkpoint] 48M x {B} envs x {steps} steps: max rel hidden error {worst_h:.3e}; "
              f"argmax tokens equal {agree}/{total}; oracle top-2 margins at the flips "
              f"{[round(m, 5) for m in flipped_margin]}")
    assert worst_h < 2e-2
    assert agree / total > 0.97
    assert all(m < 2e-2 for m in flipped_margin)        # only near-ties may flip
    eng.close()


@pytest.mark.parametrize("name,B", [("16M", 64), ("48M", 40)])
@pytest.mark.parametrize("opts", [{"up_fuse": 1}, {"state_fuse": 1}, {"state_fuse": 2}, {"up_fuse": 1, "state_fuse": 2}])
def test_chain_fusion_options_equal_default(name, B, opts):
    """The measured-and-not-default fusions of the per-block chain (pre-cell work in the proj_up epilogue; finalize
    inside the state stream kernel through a thread-block cluster per (env, head), symmetric or leader variant) compute
    the same step as the default kernels: identical action tokens, hidden states and recurrent state to rounding of
    the differently ordered partial sums."""
    cfg, sd, eng = _engine(name, B, seed=4)
    states, rtg, _ = make_stream(cfg, range(B), 4, domains="mixed", seed=31)
    res = {}
    for tag, o in (("default", {}), ("fused", opts)):
        for k in ("up_fuse", "state_fuse"):
            eng.set_option(k, o.get(k, 0))
        cache, out = eng.new_state(B), None
        s_dev = torch.empty(B, cfg.state_dim, device="cuda")
        r_dev = torch.empty(B, device="cuda")
        toks, hids = [], []
        eng.launch_count()
        for t in range(4):
            s_dev.copy_(torch.from_numpy(states[t]))
            r_dev.copy_(torch.from_numpy(rtg[t]))
            out = eng.policy_step(cache, s_dev, r_dev, flags=L.XL_FLAG_GRAPH if t else 0, want_hidden=True, out=out)
            torch.cuda.synchronize()
            toks.append(out["action_tokens"].cpu().clone())
            hids.append(out["last_hidden_state"].cpu().clone())
        last = cfg.num_blocks - 1
        res[tag] = (torch.stack(toks), torch.stack(hids), cache.view(last, L.XL_STATE_C).cpu().clone(),
                    cache.view(last, L.XL_STATE_N).cpu().clone(), cache.view(last, L.XL_STATE_CONV).cpu().clone(),
                    eng.launch_count())
    a, b = res["default"], res["fused"]
    assert torch.equal(a[0], b[0])
    assert _rel(b[1], a[1]) < 1e-4
    assert _rel(b[2], a[2]) < 1e-4 and _rel(b[3], a[3]) < 1e-4 and _rel(b[4], a[4]) < 1e-5
    assert b[5] < a[5]                                   # fewer launches: a kernel per block really disappeared
    eng.close()


# ------------------------------------------------------------------------------------------------------------
# BASELINE.md §2b, config 4: chunkwise context prefill vs SEQUENTIAL oracle stepping on an S = 3000-token prefix
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["16M", "48M"])
def test_prefill_3000_token_prefix_vs_sequential_oracle(name):
    """`xl_policy_prefill` over 1000 timesteps = 3000 tokens (s, rtg, r) of one env — chunk after chunk through the
    tensor-core sequence cell — must leave the recurrent state where 3000 sequential oracle token steps leave it
    (`xLSTMBlockStack.step` in a loop, decision_xlstm.py:161-165: the only way the reference reaches such a context),
    and the rollout that follows must produce the oracle's action tokens bit-exactly. 206M: tools/bench_prefill.py --check."""
    from oracle import xlstm_oracle as O
    Tn, Tr = 1000, 3
    cfg, sd, eng = _engine(name, 1, seed=6)
    ora = O.OraclePolicy(cfg, sd)
    states, rtg, _ = make_stream(cfg, range(1), Tn + Tr, domains="dmcontrol", seed=2024)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    cache = eng.new_state(1)
    eng.policy_prefill(cache, dev(states[:Tn].transpose(1, 0, 2)), dev(rtg[:Tn].T))
    pkv = None
    for t in range(Tn):                                   # 3000 sequential token steps on the CPU, fp32
        x = ora.embed(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), torch.zeros(1))
        _, pkv = ora.encoder.forward_cached(x, pkv)
    exp = cache.to_past_key_values()
    for i in range(cfg.num_blocks):
        c, n, m = pkv[f"block_{i}"]["mlstm_state"]
        ce, ne, me = exp[f"block_{i}"]["mlstm_state"]
        assert _rel(ce.cpu(), c) < REL_TOL and _rel(ne.cpu(), n) < REL_TOL, f"block {i}"
        assert (me.cpu() - m).abs().max() < 1e-3 * max(1.0, m.abs().max().item()), f"block {i}"
        assert _rel(exp[f"block_{i}"]["conv_state"][0].cpu(), pkv[f"block_{i}"]["conv_state"][0]) < 1e-4
    for t in range(Tn, Tn + Tr):
        out = eng.policy_step(cache, dev(states[t]), dev(rtg[t]), want_hidden=True, want_logits=True)
        ref = ora.step(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), past_key_values=pkv)
        pkv = ref["past_key_values"]
        margins = _margin_ok(ref["action_logits"], out["action_tokens"].cpu().long(), ref["action_tokens"])
        assert not margins, f"token mismatches after the prefill at t={t}: oracle top-2 margins {margins}"
        assert _rel(out["last_hidden_state"].cpu(), ref["last_hidden_state"]) < REL_TOL
    eng.close()


def test_batched_rollout_with_context_prefill():
    """BatchedRollout.prefill_context (the batched `persist_context`: a context of earlier timesteps warms the state in
    one chunkwise pass) + run(keep_state=True) == stepping through the context first and then rolling out."""
    from lram_b200.rollout import BatchedRollout
    from lram_b200.synth import SyntheticEnvBatch
    cfg, sd, eng = _engine("16M", 4, seed=8)
    Tn, Tr = 19, 5
    ctx_states, ctx_rtg, _ = make_stream(cfg, range(4), Tn, domains="mixed", seed=55)
    res = {}
    for tag in ("prefill", "stepped"):
        envs = SyntheticEnvBatch(cfg, range(4), domains="mixed", ep_len=3, seed=77)
        ro = BatchedRollout(eng, envs, use_graph=True)
        if tag == "prefill":
            ro.prefill_context(ctx_states.transpose(1, 0, 2), ctx_rtg.T)
        else:
            eng.reset(ro.state)
            for t in range(Tn):
                eng.policy_step(ro.state, torch.from_numpy(ctx_states[t]).cuda(), torch.from_numpy(ctx_rtg[t]).cuda())
        res[tag] = ro.run(Tr, record=True, keep_state=True)
    assert np.array_equal(res["prefill"]["tokens"], res["stepped"]["tokens"])
    assert np.array_equal(res["prefill"]["actions"], res["stepped"]["actions"])
    eng.close()


def test_host_step_equals_device_step():
    """`xl_policy_step_host` (host buffers in, host buffers out, graph-replayed step in between) gives the tokens /
    actions of the device-pointer entry point, step after step, with alternating pinned buffers and with pageable ones."""
    cfg, sd, eng = _engine("16M", 6, seed=2)
    states, rtg, _ = make_stream(cfg, range(6), 5, domains="mixed")
    ca, cb = eng.new_state(6), eng.new_state(6)
    bufs = [(torch.zeros(6, cfg.state_dim).pin_memory(), torch.zeros(6).pin_memory(),
             torch.zeros(6, cfg.act_dim, dtype=torch.int32).pin_memory(), torch.zeros(6, cfg.act_dim).pin_memory())
            for _ in range(2)]
    for t in range(5):
        hs, hr, ht, ha = bufs[t % 2]
        hs.copy_(torch.from_numpy(states[t]))
        hr.copy_(torch.from_numpy(rtg[t]))
        eng.policy_step_host(ca, hs, hr, ht, ha, flags=L.XL_FLAG_GRAPH)
        o = eng.policy_step(cb, torch.from_numpy(states[t]).cuda(), torch.from_numpy(rtg[t]).cuda())
        torch.cuda.synchronize()
        assert torch.equal(ht, o["action_tokens"].cpu()) and torch.equal(ha, o["action_preds"].cpu()), t
    # pageable host memory works too (synchronous staging by the driver)
    hs, hr = torch.from_numpy(states[0]).clone(), torch.from_numpy(rtg[0]).clone()
    ht, ha = torch.zeros(6, cfg.act_dim, dtype=torch.int32), torch.zeros(6, cfg.act_dim)
    cc, cd = eng.new_state(6), eng.new_state(6)
    eng.policy_step_host(cc, hs, hr, ht, ha, flags=L.XL_FLAG_GRAPH)
    o = eng.policy_step(cd, hs.cuda(), hr.cuda())
    torch.cuda.synchronize()
    assert torch.equal(ht, o["action_tokens"].cpu())
    eng.close()


def test_token_ring_single_gpu():
    """`xl_set_token_ring`: every policy step (eager or graph-replayed) also stores its tokens in the next ring slot;
    re-seeking and disarming work."""
    cfg, sd, eng = _engine("toy128", 5)
    states, rtg, _ = make_stream(cfg, range(5), 7, domains="mixed")
    ring = torch.full((4, 5, cfg.act_dim), -1, dtype=torch.int32, device="cuda")
    eng.set_token_ring(ring, 0)
    cache, out, toks = eng.new_state(5), None, []
    s_dev, r_dev = torch.empty(5, cfg.state_dim, device="cuda"), torch.empty(5, device="cuda")
    for t in range(7):
        s_dev.copy_(torch.from_numpy(states[t]))
        r_dev.copy_(torch.from_numpy(rtg[t]))
        out = eng.policy_step(cache, s_dev, r_dev, flags=L.XL_FLAG_GRAPH if t % 2 else 0, out=out)
        torch.cuda.synchronize()
        toks.append(out["action_tokens"].clone())
        assert torch.equal(ring[t % 4], toks[-1]), t
    eng.set_token_ring(ring, 2)                       # re-seek: the next step lands in slot 2
    out = eng.policy_step(cache, s_dev, r_dev, flags=L.XL_FLAG_GRAPH, out=out)
    torch.cuda.synchronize()
    assert torch.equal(ring[2], out["action_tokens"])
    eng.set_token_ring(None)
    before = ring.clone()
    eng.policy_step(cache, s_dev, r_dev, flags=L.XL_FLAG_GRAPH, out=out)
    torch.cuda.synchronize()
    assert torch.equal(ring, before)
    eng.close()


@pytest.mark.parametrize("opt,val", [("gemm_bm", 64), ("gemm_cluster", 2), ("gemm_cluster", 4)])
def test_gemm_tile_variants_bit_identical(opt, val):
    """64-row UMMA tiles (cta_group::1, M = 64: accumulator rows in lanes 0-15 of each TMEM quarter) and the A-tile TMA
    multicast across a cluster of column-tile CTAs compute exactly the plain tcgen05 Linear: same products, same order."""
    cfg, sd, eng = _engine("toy", 1)
    g = torch.Generator().manual_seed(5)
    try:
        for (M, N, K) in [(192, 3072, 768), (192, 768, 1536), (100, 640, 256), (33, 128, 64)]:
            A = torch.randn(M, K, generator=g).cuda()
            W = (torch.randn(N, K, generator=g) * 0.05).to(torch.bfloat16).cuda()
            bias = torch.randn(N, generator=g).cuda()
            eng.set_option(opt, 0 if opt == "gemm_bm" else 1)
            ref = eng.linear(A, W, bias, None, impl=2)
            eng.set_option(opt, val)
            out = eng.linear(A, W, bias, None, impl=2)
            torch.cuda.synchronize()
            assert torch.equal(out, ref), (opt, val, M, N, K)
            ref64 = (A.double() @ W.double().t() + bias.double()).float()
            assert _rel(out, ref64) < 2e-5
    finally:
        eng.set_option(opt, 0 if opt == "gemm_bm" else 1)      # process-wide switches: restore
        eng.close()


def test_gemm_2sm_pair_bit_identical():
    """2-SM Linear (option "gemm_2cta": a CTA pair computes a 256 x 256 tile with tcgen05.mma.cta_group::2, each CTA
    staging its 128 rows of the A planes and half of the W tile) == the 1-SM tcgen05 Linear bit for bit (same products in
    the same order), incl. ragged M / N edges, bias and residual."""
    cfg, sd, eng = _engine("toy", 1)
    g = torch.Generator().manual_seed(7)
    try:
        # (the last shape has 160 tiles: more than the 74 CTA pairs, so the persistent variant walks 2-3 tiles per pair)
        for (M, N, K) in [(1000, 2560, 768), (640, 1280, 1024), (600, 2192, 512), (512, 256, 64), (1300, 768, 640),
                          (4000, 2560, 256)]:
            A = torch.randn(M, K, generator=g).cuda()
            W = (torch.randn(N, K, generator=g) * 0.05).to(torch.bfloat16).cuda()
            bias = torch.randn(N, generator=g).cuda()
            res = torch.randn(M, N, generator=g).cuda()
            eng.set_option("gemm_2cta", 0)
            ref = eng.linear(A, W, bias, res, impl=2)
            for variant in (1, 2):        # 1 = one tile per CTA pair, 2 = persistent pairs, double-buffered TMEM accumulator
                eng.set_option("gemm_2cta", variant)
                out = eng.linear(A, W, bias, res, impl=2)
                torch.cuda.synchronize()
                assert torch.equal(out, ref), (variant, M, N, K, (out - ref).abs().max().item())
            ref64 = (A.double() @ W.double().t() + bias.double() + res.double()).float()
            assert _rel(out, ref64) < 2e-5
    finally:
        eng.set_option("gemm_2cta", -1)      # process-wide switch: restore the default
        eng.close()


def test_argmax_head_edge_cases_match_torch_semantics():
    """The fused argmax / inv_tokenize kernel on crafted logits (head weight 0, so logits == bias exactly): ties take the
    FIRST index and NaN counts as the maximum (torch.argmax, multi_domain_discrete_dt_model.py:83-94); ids below the
    tokenizer shift decode to min_val (minmax_tokenizer.py:34-37); the discrete branch only looks at the first 18 logits."""
    from lram_b200.engine import XLSTMEngine
    from oracle.xlstm_oracle import OracleMinMaxTokenizer
    cfg = preset("toy")
    sd = make_state_dict(cfg, seed=1)
    sd["action_net.0.weight"] = torch.zeros_like(sd["action_net.0.weight"])
    g = torch.Generator().manual_seed(0)
    bias = torch.randn(cfg.act_dim, cfg.num_actions, generator=g)
    bias[0, :] = 0.25                                   # all equal -> token 0
    bias[1, 17] = 9.0                                   # id below the shift -> decodes to -1.0
    bias[2, 18] = 9.0                                   # first continuous bin
    bias[3, 273] = 9.0                                  # last bin
    bias[4, 100] = float("nan")                         # NaN is the maximum
    bias[5, 200] = float("nan"); bias[5, 50] = float("nan")     # first NaN wins
    bias[6, 40] = 7.0; bias[6, 30] = 7.0                # tie -> first
    bias[7, :] = -float("inf"); bias[7, 60] = -1e30     # -inf everywhere else
    sd["action_net.0.bias"] = bias.reshape(-1).clone()
    eng = XLSTMEngine(cfg, sd, max_batch=3)
    states, rtg, _ = make_stream(cfg, range(3), 1, domains="mixed")
    out = eng.policy_step(eng.new_state(3), torch.from_numpy(states[0]).cuda(), torch.from_numpy(rtg[0]).cuda(),
                          want_logits=True)
    torch.cuda.synchronize()
    lg = out["action_logits"].cpu().view(3, cfg.act_dim, cfg.num_actions)
    assert torch.equal(torch.nan_to_num(lg[0], nan=123.0), torch.nan_to_num(bias, nan=123.0))     # logits == bias, bit for bit
    ref_tok = torch.argmax(lg, dim=-1)
    assert ref_tok[0].tolist() == [0, 17, 18, 273, 100, 50, 30, 60]
    assert torch.equal(out["action_tokens"].cpu().long(), ref_tok)
    ref_act = OracleMinMaxTokenizer(cfg.action_channels, cfg.discrete_actions).inv_tokenize(ref_tok)
    assert torch.equal(out["action_preds"].cpu(), ref_act)
    assert ref_act[0, :3].tolist() == [-1.0, -1.0, -1.0] and ref_act[0, 3].item() == 255 * (2.0 / 256) - 1.0
    # discrete branch: argmax over logits[:18] of the first action dimension only
    bias_d = bias.clone()
    bias_d[0, :] = torch.randn(cfg.num_actions, generator=g)
    bias_d[0, 20] = 50.0                                # the global maximum sits outside the 18 discrete actions
    bias_d[0, 5] = 10.0
    sd["action_net.0.bias"] = bias_d.reshape(-1).clone()
    eng2 = XLSTMEngine(cfg, sd, max_batch=3)
    out = eng2.policy_step(eng2.new_state(3), torch.from_numpy(states[0]).cuda(), torch.from_numpy(rtg[0]).cuda(),
                           flags=L.XL_FLAG_DISCRETE)
    torch.cuda.synchronize()
    assert out["action_tokens"].cpu()[:, 0].tolist() == [5, 5, 5]
    eng.close(); eng2.close()
