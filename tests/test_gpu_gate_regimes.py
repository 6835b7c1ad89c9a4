"""Every mLSTM cell against the float64 reference at the gate extremes (run on the B200: pytest -m gpu).

The scenarios, the float64 reference and the comparison rule live in tests/test_gate_regimes_reference.py, whose CPU
tests check that each scenario reaches its regime and that the bound is reachable. The rule, for every test here:
  * state: per (env, head) max|dC| / max|C_ref| of that head, likewise n, within BOUND (1e-4); m absolutely within
    M_BOUND of max(1, |m|) (|m|: the largest of the head so far, see m_err);
  * per-token outputs: h (from num, qn, m) and the finalize output per (env, head, token) row against that row's own
    maximum, within BOUND plus the rounding of the row's sums under cancellation: u kappa (see U_FP32 / U_TC);
  * every output finite.
The worst errors per cell and scenario are printed (pytest -s) under the tag GATE-REGIME.
"""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_gate_regimes_reference as R  # noqa: E402

from lram_b200.config import preset  # noqa: E402
from lram_b200.synth import make_state_dict  # noqa: E402

DEFAULT_PREFILL_CELL, DEFAULT_STATE_IMPL = 2, 1      # library defaults of xl_set_option "prefill_cell" / "state_impl"
PRESET_OF_DH = {32: "toy", 64: "toy128", 256: "16M", 384: "48M", 512: "110M", 640: "206M"}
CELL_NAMES = {0: "fp32", 1: "mma.sync", 2: "tcgen05"}
CELL_DHS = {0: [32, 64, 256, 384, 512, 640], 1: [32, 64, 256, 384, 512, 640], 2: [256, 384, 512, 640]}


@pytest.fixture(scope="module")
def engines():
    from lram_b200.engine import XLSTMEngine
    made = {}

    def get(DH):
        if DH not in made:
            cfg = preset(PRESET_OF_DH[DH], num_blocks=1)
            assert cfg.head_dim == DH and cfg.num_heads == R.NH
            made[DH] = XLSTMEngine(cfg, make_state_dict(cfg, seed=0), max_batch=2)
        return made[DH]

    yield get
    for eng in made.values():
        eng.close()


def _report(tag, errs):
    print(f"GATE-REGIME {tag}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()), flush=True)


def _check(errs, ratios):
    """errs: state and m errors (bounds BOUND / M_BOUND); ratios: per-row output errors over their row's bound."""
    for k, e in errs.items():
        if k.startswith(("C", "n", "m")):
            assert e <= (R.M_BOUND if k.startswith("m") else R.BOUND), (k, e)
    for k, r in ratios.items():
        assert r <= 1.0, (k, r)


def _state_errs(errs, C, n, m, ref_state, m_scale, at):
    Cr, nr, mr = ref_state
    for x in (C, n, m):
        assert torch.isfinite(x).all(), at
    errs[f"C@{at}"] = max(errs.get(f"C@{at}", 0.0), R.head_rel(C.cpu(), Cr))
    errs[f"n@{at}"] = max(errs.get(f"n@{at}", 0.0), R.head_rel(n.cpu(), nr))
    errs[f"m@{at}"] = max(errs.get(f"m@{at}", 0.0), R.m_err(m.cpu(), mr, m_scale))


# ---- (a) the sequence cells through xl_mlstm_cell_seq ---------------------------------------------------------------
SEQ_CASES = [(name, DH, cell) for name in R.SCENARIOS for DH in (32, 64, 256, 384, 512, 640) for cell in (0, 1, 2)
             if DH in CELL_DHS[cell]]


@pytest.mark.parametrize("name,DH,cell", SEQ_CASES)
def test_cell_seq_gate_regimes(engines, name, DH, cell):
    """Two consecutive calls (the second continues from the carried state) of the cell `prefill_cell` selects, lengths
    that end in a ragged stage / chunk, against the float64 recurrence."""
    sc = R.SCENARIOS[name]
    inp, ref = R.reference(name, DH)
    eng = engines(DH)
    eng.set_option("prefill_cell", cell)
    try:
        errs, ratios = _run_cell_seq(eng, sc, inp, ref, DH, cell)
    finally:
        eng.set_option("prefill_cell", DEFAULT_PREFILL_CELL)
    _report(f"seq cell={CELL_NAMES[cell]} {name} DH={DH}", {**errs, **{f"{k}/bound": v for k, v in ratios.items()}})
    _check(errs, ratios)


def _run_cell_seq(eng, sc, inp, ref, DH, cell):
    B, dev = sc.B, eng.device
    C, n, m = inp["C0"].to(dev), inp["n0"].to(dev), inp["m0"].to(dev)
    w, skip = inp["outnorm_w"].to(dev), inp["skip"].to(dev)
    errs, ratios = {}, {"h": 0.0, "out": 0.0}
    for t0, t1 in R.calls(sc, cell):
        S = t1 - t0

        def rows(x):
            return x[:, t0:t1].reshape(B * S, -1).contiguous().to(dev)

        gates = rows(torch.stack([inp["ig"], inp["fg"]], 2))
        u = rows(torch.cat([torch.zeros_like(inp["z"]), inp["z"]], -1))
        num, qn, mseq, out, which = eng.cell_seq(C, n, m, rows(inp["q"]), rows(inp["k"]), rows(inp["v"]), gates,
                                                 rows(inp["act"]), u, w, skip, B, S)
        torch.cuda.synchronize()
        assert which == cell, f"asked for the {CELL_NAMES[cell]} cell, {CELL_NAMES.get(which)} ran"
        for x in (num, qn, mseq, out):
            assert torch.isfinite(x).all(), f"non-finite output over tokens [{t0}, {t1})"
        m_h = mseq.cpu().view(B, R.NH, S)
        h = R.h_of(R.heads_rows(num.cpu(), B, S), qn.cpu().view(B, S, R.NH).transpose(1, 2), m_h)
        tol = R.BOUND + (R.U_FP32 if cell == 0 else R.U_TC) * ref["kappa"][..., t0:t1]
        eh, rh = R.row_rel(h, ref["h"][:, :, t0:t1], tol)
        eo, ro = R.row_rel(R.heads_rows(out.cpu(), B, S), R.heads_rows(ref["out"][:, t0:t1], B, S), tol)
        errs["h"], errs["out"] = max(errs.get("h", 0.0), eh), max(errs.get("out", 0.0), eo)
        ratios["h"], ratios["out"] = max(ratios["h"], rh), max(ratios["out"], ro)
        errs["m"] = max(errs.get("m", 0.0), R.m_err(m_h, ref["m"][..., t0:t1], ref["m_scale"][..., t0:t1]))
        _state_errs(errs, C, n, m, ref["states"][t1], ref["m_scale"][..., t1 - 1], "call")
    return errs, ratios


def test_cell_seq_rejects_a_shape_its_cell_cannot_take(engines):
    """The requested cell does not fall back: S % 16 != 0 on the mma.sync cell, S < 64 on the tcgen05 cell."""
    from lram_b200 import _lib as L
    eng = engines(256)
    dev, B, inner, NH = eng.device, 1, 1024, R.NH
    try:
        for cell, S in ((1, 24), (2, 48)):
            eng.set_option("prefill_cell", cell)
            z = torch.zeros(B * S, inner, device=dev)
            C, n, m = (torch.zeros(B, NH, 256, 256, device=dev), torch.zeros(B, NH, 256, device=dev),
                       torch.zeros(B, NH, device=dev))
            with pytest.raises(L.XLError) as ei:
                eng.cell_seq(C, n, m, z, z, z, torch.zeros(B * S, 2 * NH, device=dev), z,
                             torch.zeros(B * S, 2 * inner, device=dev), z[0], z[0], B, S)
            assert ei.value.code == L.XL_ERR_UNSUPPORTED
    finally:
        eng.set_option("prefill_cell", DEFAULT_PREFILL_CELL)


# ---- (b) the step cell through xl_mlstm_cell_step -------------------------------------------------------------------
STEP_CASES = [(name, DH, T, impl) for name in R.SCENARIOS for DH in (64, 256) for T in (1, 2, 3, 4)
              for impl in (0, 1, 2)]


@pytest.mark.parametrize("name,DH,T,impl", STEP_CASES)
def test_cell_step_gate_regimes(engines, name, DH, T, impl):
    """Every token of the scenario through the step cell, T tokens per launch (the remainder in a last, shorter one),
    against the float64 recurrence: h_raw, h_norm per row, the state after the last token."""
    from lram_b200.engine import c_from_slab, c_to_slab
    from oracle import xlstm_oracle as O
    sc = R.SCENARIOS[name]
    inp, ref = R.reference(name, DH)
    eng = engines(DH)
    eng.set_option("state_impl", impl)
    B, inner, dev = sc.B, R.NH * DH, eng.device
    N = sc.base + R.TAIL
    C, n, m = c_to_slab(inp["C0"]).to(dev), inp["n0"].to(dev), inp["m0"].to(dev)
    w = inp["outnorm_w"].to(dev)
    qkv = torch.stack([inp["q"], inp["k"], inp["v"]], 2).reshape(B, N, 3, inner).to(dev)
    ig, fg = inp["ig"].to(dev), inp["fg"].to(dev)
    h_raw, h_norm = torch.empty(B, N, inner, device=dev), torch.empty(B, N, inner, device=dev)
    t = 0
    try:
        while t < N:
            Tl = min(T, N - t)
            hn, hr = eng.cell_step(C, n, m, qkv[:, t:t + Tl].reshape(B * Tl, 3, inner).contiguous(),
                                   ig[:, t:t + Tl].reshape(B * Tl, R.NH).contiguous(),
                                   fg[:, t:t + Tl].reshape(B * Tl, R.NH).contiguous(), w, B, Tl, slab=True)
            h_raw[:, t:t + Tl] = hr.view(B, Tl, inner)
            h_norm[:, t:t + Tl] = hn.view(B, Tl, inner)
            t += Tl
        torch.cuda.synchronize()
    finally:
        eng.set_option("state_impl", DEFAULT_STATE_IMPL)
    for x in (h_raw, h_norm):
        assert torch.isfinite(x).all()
    tol = R.BOUND + R.U_FP32 * ref["kappa"]
    hn_ref = O.multihead_layer_norm(ref["h"], inp["outnorm_w"].double(), eps=R.LN_EPS)
    errs, ratios = {}, {}
    errs["h"], ratios["h"] = R.row_rel(R.heads_rows(h_raw.cpu(), B, N), ref["h"], tol)
    errs["h_norm"], ratios["h_norm"] = R.row_rel(R.heads_rows(h_norm.cpu(), B, N), hn_ref, tol)
    _state_errs(errs, c_from_slab(C), n, m, ref["states"][N], ref["m_scale"][..., N - 1], N)
    _report(f"step T={T} impl={impl} {name} DH={DH}", {**errs, **{f"{k}/bound": v for k, v in ratios.items()}})
    _check(errs, ratios)


# ---- (c) end to end: context prefill, then steps, on gate-heavy weights ---------------------------------------------
E2E_CASES = [("toy128", 1, False), ("toy128", 1, True), ("toy128", 0, False), ("toy128", 0, True),
             ("16M", 2, False), ("16M", 2, True), ("toy128-ms", 1, False)]


def _mlstm_blocks(cfg):
    return [i for i in range(cfg.num_blocks) if not cfg.is_slstm(i)]


def _compare_env_state(cfg, got, ref, m_hist, ig_abs, errs):
    """One env's past_key_values (GPU export vs float64 oracle): C, n per head; m against the largest |m| of its head
    (m_hist [tokens, mLSTM blocks, NH]) plus the rounding of the input-gate projection m takes over at every reset,
    U_FP32 sum_j |w_j g_j| (ig_abs, same shape; the unit tests feed exact gates and have no such term); the conv
    window per block; the sLSTM planes per (plane, head)."""
    for j, i in enumerate(_mlstm_blocks(cfg)):
        (c, n, m), (cr, nr, mr) = got[f"block_{i}"]["mlstm_state"], ref[f"block_{i}"]["mlstm_state"]
        scale = torch.cat([m_hist[:, j], mr.view(1, -1)]).abs().amax(0).clamp_min(1.0)
        scale = scale + R.U_FP32 / R.M_BOUND * ig_abs[:, j].amax(0)
        errs["C"] = max(errs.get("C", 0.0), R.head_rel(c.cpu(), cr))
        errs["n"] = max(errs.get("n", 0.0), R.head_rel(n.cpu(), nr))
        errs["m"] = max(errs.get("m", 0.0), R.m_err(m.cpu().view(-1), mr.view(-1), scale))
    for i in range(cfg.num_blocks):
        g, r = got[f"block_{i}"], ref[f"block_{i}"]
        cg, cr = g["conv_state"][0].cpu(), r["conv_state"][0]
        errs["conv"] = max(errs.get("conv", 0.0), R.head_rel(cg.reshape(1, 1, -1), cr.reshape(1, 1, -1)))
        if cfg.is_slstm(i):
            sg, sr = g["slstm_state"].cpu().reshape(4, R.NH, -1), r["slstm_state"].reshape(4, R.NH, -1)
            errs["slstm"] = max(errs.get("slstm", 0.0), R.head_rel(sg, sr))


@pytest.mark.parametrize("name,cell,ragged", E2E_CASES)
def test_prefill_then_steps_on_gate_heavy_weights(name, cell, ragged):
    """XLSTMEngine.prefill (uniform, or lengths= with one env at 0 and one short) then 3 step-path tokens from the
    prefilled state, against the float64 OracleEncoder stepped token by token: hidden rows of the prefill and of the
    steps per (env, token) within BOUND + U_TC kappa (kappa: the largest over the token's mLSTM heads; the Linear
    layers multiply bf16 hi/lo operands too), and every part of every block's state. The recorded gates must reach
    scenarios 2, 4 and 5 in every mLSTM block."""
    from lram_b200.engine import XLSTMEngine
    cfg = preset(name, num_blocks=2) if name == "16M" else preset(name)
    sd = R.gate_heavy_state_dict(cfg)
    B, S = 3, 392                            # 3 x 128 + 8: a ragged last chunk of every cell
    lengths = [S, 0, 37] if ragged else None
    g = torch.Generator().manual_seed(9)
    x, xs = torch.randn(B, S, cfg.d, generator=g), torch.randn(B, 3, cfg.d, generator=g)
    eng = XLSTMEngine(cfg, sd, max_batch=B)
    try:
        eng.set_option("prefill_cell", cell)
        cache = eng.new_state(B)
        hid = eng.prefill(cache, x.cuda(), lengths=lengths).cpu()
        steps = torch.cat([eng.encoder_step(cache, xs[:, t:t + 1].contiguous().cuda()).cpu() for t in range(3)], 1)
        torch.cuda.synchronize()
        exported = cache.to_past_key_values()
    finally:
        eng.close()
    for t in (hid, steps):
        assert torch.isfinite(t).all()
    ora = R.oracle64(cfg, sd)
    lens = lengths or [S] * B
    errs, ratios, recs = {}, {"hidden": 0.0, "step": 0.0}, []
    for b in range(B):
        pkv, m_hist, ig_abs = None, [], []
        if lens[b]:
            y, pkv, rec = R.run_oracle_recorded(ora, x[b:b + 1, :lens[b]].double())
            recs.append(rec)
            m_hist.append(rec["m"][:, :, 0])
            ig_abs.append(rec["ig_abs"][:, :, 0])
            tol = R.BOUND + R.U_TC * rec["kappa"][:, :, 0].amax((1, 2))
            e, r = R.row_rel(hid[b, :lens[b]], y[0], tol)
            errs["hidden"], ratios["hidden"] = max(errs.get("hidden", 0.0), e), max(ratios["hidden"], r)
        assert torch.all(hid[b, lens[b]:] == 0), f"env {b}: rows past its length"
        ys, pkv, rec = R.run_oracle_recorded(ora, xs[b:b + 1].double(), pkv)
        m_hist.append(rec["m"][:, :, 0])
        ig_abs.append(rec["ig_abs"][:, :, 0])
        tol = R.BOUND + R.U_TC * rec["kappa"][:, :, 0].amax((1, 2))
        e, r = R.row_rel(steps[b], ys[0], tol)
        errs["step"], ratios["step"] = max(errs.get("step", 0.0), e), max(ratios["step"], r)
        env = {k: {kk: (tuple(t[b:b + 1] for t in vv) if kk == "mlstm_state" else
                        (vv[:, b:b + 1] if kk == "slstm_state" else (vv[0][b:b + 1],)))
                   for kk, vv in v.items()} for k, v in exported.items()}
        _compare_env_state(cfg, env, pkv, torch.cat(m_hist), torch.cat(ig_abs), errs)
    R.assert_gate_heavy_coverage(recs[0], name)                         # env 0 runs the whole context
    _report(f"e2e {name} cell={CELL_NAMES[cell]} {'ragged' if ragged else 'uniform'}",
            {**errs, **{f"{k}/bound": v for k, v in ratios.items()}})
    _check({k: v for k, v in errs.items() if k in ("C", "n", "m")}, ratios)
    for k in ("conv", "slstm"):
        assert errs.get(k, 0.0) <= R.BOUND, (k, errs[k])
