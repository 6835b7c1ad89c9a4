"""Gate regimes of the mLSTM cell and their float64 reference (CPU only).

Trained xLSTM checkpoints leave the narrow gate window of the synthetic weights (lram_b200/synth.py): heads that
forget almost everything every token, input gates that spike by tens, a stabiliser m far below zero. The cells have
code for exactly these regimes (the fp32 sequence cell's plain-recurrence stages when a stage's decay F_8 < 1e-12, the
-200 log clamp of the chunkwise cells when the stabilised forget gate underflows, the gate scan's composition of
2048-token super-chunks). This module names one gate scenario per regime, builds its q / k / v / gates as plain
tensors, and runs the oracle's recurrence (oracle.xlstm_oracle.recurrent_step_stabilized_simple) in float64 as the
reference that tests/test_gpu_gate_regimes.py compares every cell with.

Here, on the CPU: each scenario must reach the regime it claims (computed from the float64 reference alone), and the
plain fp32 oracle must meet the GPU tests' per-head / per-row bound against the float64 reference on every scenario,
so that the bound is known to be reachable.
"""
from __future__ import annotations

import functools
import math
from dataclasses import dataclass
from typing import Dict, Tuple

import pytest
import torch
import torch.nn.functional as F

from oracle import xlstm_oracle as O

NH = 4                       # every preset has 4 heads
LN_EPS, CELL_EPS = 1e-5, 1e-6
BOUND = 1e-4                 # per-head (state) / per-row (outputs) relative bound of every comparison here
# A row's h = num / den also carries the rounding of the sums behind num = q^T C and q.n, ill-conditioned where they
# cancel: with |C|^ and |n|^ the states of absolute values (C^ <- f C^ + i |k| |v|^T), |d num_j| <= u (|q|^T |C|^)_j and
# |d den| <= u |q|^T |n|^, u the relative rounding of one product term. So the row's bound is BOUND + u kappa with
# kappa = max_j (|q|^T |C|^)_j / max_j |num_j| + |q|^T |n|^ / den. u = U_FP32 for fp32 arithmetic (fp32 oracle: at most
# 3.1e-6 kappa here, the state's own accumulated rounding included), U_TC where the operands are bf16 hi/lo pairs (two
# 2^-17 splits per product).
U_FP32 = 2.0 ** -18
U_TC = 2.0 ** -15
LOG_MIN_DECAY = math.log(1e-12)   # the fp32 sequence cell's kMinDecay: below it a stage runs the plain recurrence
EXPF_UNDERFLOW = -104.0      # float32 expf(x) == 0 for x below about -103.97
TAIL = 88                    # tokens after `base`: room for the second call of every cell (see calls())


@dataclass(frozen=True)
class Scenario:
    name: str
    seed: int
    base: int                # tokens of the first call of the fp32 / tcgen05 cells (mma.sync: base + 8)
    B: int
    regime: str


SCENARIOS = {s.name: s for s in (
    Scenario("mild", 11, 296, 2, "today's synthetic window: fgate bias 3..6, input gates near 0 (control)"),
    Scenario("strong_forget", 12, 296, 2, "fg ~ N(-4, 1): stage decays far below 1e-12, the exp(-m) denominator"),
    Scenario("straddle", 13, 296, 2, "per-head fg near -3.42: 8-token stage decays on both sides of 1e-12"),
    Scenario("spikes", 14, 296, 2, "ig ~ -10 with +60..+100 spikes at stage / chunk / call edges: f underflows"),
    Scenario("negative_m", 15, 296, 2, "ig ~ -30, fg ~ +2, carried m0 = -50: m far below zero"),
    Scenario("long_memory", 16, 2312, 1, "fg ~ +12 over > 2048 tokens: the gate scan composes super-chunks"),
)}


def calls(sc: Scenario, cell: int) -> Tuple[Tuple[int, int], Tuple[int, int]]:
    """Token ranges of the two consecutive calls a cell runs (the second continues from the carried state).
    fp32 (0) and tcgen05 (2): base + 72 tokens, base % 16 == 8 and no length a multiple of 128 (ragged last stage /
    chunk); mma.sync (1): lengths multiples of its 16-token chunk, still not of 128."""
    n1, n2 = (sc.base + 8, 80) if cell == 1 else (sc.base, 72)
    return (0, n1), (n1, n1 + n2)


def spike_positions(sc: Scenario):
    """Stage and chunk edges of the three cells (8 / 16 / 128 tokens), the first token of each cell's second call and
    the last token of each second call; the `big` ones are large enough that f underflows when m sits at the
    baseline (not when a spike just before still holds m up: 8 after 7, 16 after 15, ...)."""
    b = sc.base
    big = [0, 15, 127, b, b + 8, b + 87]
    other = [7, 8, 16, 128, b + 71]
    return big, other


def make_inputs(sc: Scenario, DH: int) -> Dict[str, torch.Tensor]:
    """float32 inputs of a scenario: q, k, v [B, N, NH, DH]; ig, fg [B, N, NH] (pre-activations, bias included);
    carried C0 [B, NH, DH, DH] (reference layout), n0 [B, NH, DH], m0 [B, NH]; finalize operands act, z [B, N, NH*DH],
    outnorm_w, skip [NH*DH]. N = base + TAIL."""
    g = torch.Generator().manual_seed(sc.seed * 1000 + DH)
    B, N = sc.B, sc.base + TAIL

    def rn(*shape):
        return torch.randn(*shape, generator=g, dtype=torch.float32)

    q, k, v = rn(B, N, NH, DH), rn(B, N, NH, DH), rn(B, N, NH, DH)
    C0, n0 = rn(B, NH, DH, DH) * 0.1, rn(B, NH, DH) * 0.1
    m0 = torch.zeros(B, NH)
    noise = rn(B, N, NH)
    if sc.name == "mild":
        ig = 0.2 * rn(B, N, NH)
        fg = torch.linspace(3.0, 6.0, NH) + 0.2 * noise
        m0 = 0.3 * rn(B, NH)
    elif sc.name == "strong_forget":
        ig = rn(B, N, NH)
        fg = -4.0 + noise
    elif sc.name == "straddle":
        # a constant input gate keeps m constant, so a stage's stabilised decay is the product of the 8 forget gates:
        # 8 logsigmoid(-3.42) = log(1e-12); the heads sit 0.1 apart around it, the noise moves single stages
        ig = 0.01 * rn(B, N, NH)
        fg = torch.tensor([-3.50, -3.44, -3.40, -3.34]) + 0.02 * noise
    elif sc.name == "spikes":
        ig = -10.0 + 0.5 * rn(B, N, NH)
        big, other = spike_positions(sc)
        ig[:, big] = 96.0 + 4.0 * torch.rand(B, len(big), NH, generator=g)
        ig[:, other] = 60.0 + 40.0 * torch.rand(B, len(other), NH, generator=g)
        fg = torch.tensor([3.0, -1.0, -6.0, -16.0]) + 0.5 * noise
        m0 = torch.full((B, NH), -10.0)
    elif sc.name == "negative_m":
        ig = -30.0 + 0.5 * rn(B, N, NH)
        fg = 2.0 + 0.5 * noise
        m0 = torch.full((B, NH), -50.0)
    elif sc.name == "long_memory":
        ig = 2.0 * rn(B, N, NH)
        fg = 12.0 + 0.5 * noise
    else:
        raise KeyError(sc.name)
    inner = NH * DH
    return dict(q=q, k=k, v=v, ig=ig.contiguous(), fg=fg.contiguous(), C0=C0, n0=n0, m0=m0,
                act=rn(B, N, inner), z=rn(B, N, inner), outnorm_w=0.1 * rn(inner), skip=1.0 + 0.1 * rn(inner))


def finalize(h: torch.Tensor, act: torch.Tensor, z: torch.Tensor, outnorm_w: torch.Tensor, skip: torch.Tensor):
    """(MultiHeadLayerNorm(h) + skip * a) * silu(z): h [B, NH, S, DH]; act, z [B, S, inner] -> [B, S, inner]."""
    B, nh, S, DH = h.shape
    hn = O.multihead_layer_norm(h, outnorm_w.to(h.dtype), eps=LN_EPS).transpose(1, 2).reshape(B, S, nh * DH)
    return (hn + skip.to(h.dtype) * act.to(h.dtype)) * F.silu(z.to(h.dtype))


def gate_trace(inp, dtype=torch.float64):
    """The gate recurrence alone (m, n and the denominators need no C): per token m' [B, NH, N], the stabilised log
    forget gate lf + m - m' and whether |q.n| < exp(-m') (the exp(-m) denominator branch)."""
    ig, fg = inp["ig"].to(dtype), inp["fg"].to(dtype)
    B, N, nh = ig.shape
    DH = inp["q"].shape[-1]
    m, n = inp["m0"].to(dtype), inp["n0"].to(dtype)
    k, q = inp["k"].to(dtype) / math.sqrt(DH), inp["q"].to(dtype)
    ms, lfs, exp_branch = [], [], []
    for t in range(N):
        lf = F.logsigmoid(fg[:, t])
        mn = torch.maximum(lf + m, ig[:, t])
        lfs.append(lf + m - mn)
        n = torch.exp(lf + m - mn).unsqueeze(-1) * n + torch.exp(ig[:, t] - mn).unsqueeze(-1) * k[:, t]
        exp_branch.append((q[:, t] * n).sum(-1).abs() < torch.exp(-mn))
        m = mn
        ms.append(m)
    return torch.stack(ms, -1), torch.stack(lfs, -1), torch.stack(exp_branch, -1)


def run_reference(inp, dtype=torch.float64, checkpoints=()):
    """The oracle recurrence over all N tokens in `dtype`: h [B, NH, N, DH], m [B, NH, N], finalize output
    [B, N, inner], and the state (C [B,NH,DH,DH], n [B,NH,DH], m [B,NH]) after each token count in `checkpoints`."""
    q, k, v = (inp[x].to(dtype).transpose(1, 2) for x in ("q", "k", "v"))     # [B, NH, N, DH]
    ig, fg = (inp[x].to(dtype).transpose(1, 2) for x in ("ig", "fg"))        # [B, NH, N]
    B, nh, N, DH = q.shape
    c = inp["C0"].to(dtype).clone()
    n = inp["n0"].to(dtype).clone().unsqueeze(-1)
    m = inp["m0"].to(dtype).clone().view(B, nh, 1, 1)
    ca, na = c.abs(), n.abs()                                               # states of absolute values (kappa)
    hs, ms, kap, states = [], [], [], {}
    for t in range(N):
        qt, kt, vt = q[:, :, t:t + 1], k[:, :, t:t + 1], v[:, :, t:t + 1]
        igt, fgt = ig[:, :, t].view(B, nh, 1, 1), fg[:, :, t].view(B, nh, 1, 1)
        m_prev = m
        h, (c, n, m) = O.recurrent_step_stabilized_simple(c, n, m, qt, kt, vt, igt, fgt, eps=CELL_EPS)
        hs.append(h.squeeze(2))
        ms.append(m.view(B, nh))
        f, i = torch.exp(F.logsigmoid(fgt) + m_prev - m), torch.exp(igt - m)
        ka = kt.abs().transpose(-1, -2) / math.sqrt(DH)
        ca = f * ca + i * (ka @ vt.abs())
        na = f * na + i * ka
        den = torch.maximum((qt @ n).abs(), torch.exp(-m)) + CELL_EPS
        num_max = (qt @ c).abs().amax(-1, keepdim=True).clamp_min(1e-300)
        kap.append(((qt.abs() @ ca).amax(-1, keepdim=True) / num_max + (qt.abs() @ na) / den).view(B, nh))
        if t + 1 in checkpoints:
            states[t + 1] = (c.clone(), n.squeeze(-1).clone(), m.view(B, nh).clone())
    h = torch.stack(hs, 2)
    out = finalize(h, inp["act"], inp["z"], inp["outnorm_w"], inp["skip"])
    kappa = torch.stack(kap, -1)
    ms = torch.stack(ms, -1)
    m_scale = torch.cat([inp["m0"].to(dtype).unsqueeze(-1), ms], -1).abs().cummax(-1).values[..., 1:].clamp_min(1.0)
    return dict(h=h, m=ms, out=out, states=states, kappa=kappa, m_scale=m_scale)


@functools.lru_cache(maxsize=2)
def reference(name: str, DH: int):
    """float64 reference of a scenario at head dim DH, with the states after every call boundary of every cell."""
    sc = SCENARIOS[name]
    inp = make_inputs(sc, DH)
    cps = sorted({t for cell in (0, 1, 2) for rng in calls(sc, cell) for t in rng if t})
    return inp, run_reference(inp, torch.float64, cps)


# ---- comparison rule (shared with tests/test_gpu_gate_regimes.py) -------------------------------------------------
def head_rel(got: torch.Tensor, ref: torch.Tensor) -> float:
    """max over (env, head) of max|got - ref| / max|ref| of that head; tensors [B, NH, ...]."""
    got, ref = got.double(), ref.double()
    d = (got - ref).abs().flatten(2).amax(-1)
    s = ref.abs().flatten(2).amax(-1).clamp_min(1e-300)
    return (d / s).max().item()


def row_rel(got: torch.Tensor, ref: torch.Tensor, tol: torch.Tensor) -> Tuple[float, float]:
    """Per row (the last dim is the row): e = max|got - ref| / max|ref| of that row. Returns (max e, max e / tol), tol
    the row's bound (the reference's h_tol, shaped as the rows)."""
    got, ref = got.double(), ref.double()
    d = (got - ref).abs().amax(-1)
    e = d / ref.abs().amax(-1).clamp_min(1e-300)
    return e.max().item(), (e / tol).max().item()


def heads_rows(x: torch.Tensor, B: int, S: int) -> torch.Tensor:
    """[B*S, NH*DH] or [B, S, NH*DH] rows ([env][token]) -> [B, NH, S, DH]: one row per (env, head, token)."""
    return x.reshape(B, S, NH, -1).transpose(1, 2)


M_BOUND = 1e-5


def m_err(got: torch.Tensor, ref: torch.Tensor, scale: torch.Tensor) -> float:
    """max of |got - ref| / scale: m is compared absolutely, against M_BOUND of max(1, |m|) -- of the largest |m| of
    the head so far (the reference's m_scale): m sums forget-gate logs onto the m it decays from, so a head whose m
    came down from a spike at ~100 carries the rounding of sums at that magnitude."""
    got, ref = got.double(), ref.double()
    return ((got - ref).abs() / scale).max().item()


def h_of(num: torch.Tensor, qn: torch.Tensor, m: torch.Tensor) -> torch.Tensor:
    """h = num / (max(|qn|, exp(-m)) + eps) in float64: num [..., DH], qn and m [...]."""
    num, qn, m = num.double(), qn.double(), m.double()
    return num / (torch.maximum(qn.abs(), torch.exp(-m)) + CELL_EPS).unsqueeze(-1)


def stage_log_decay(lf_stab: torch.Tensor, lo: int, hi: int) -> torch.Tensor:
    """log F_8 of every whole 8-token stage of tokens [lo, hi) (lf_stab [B, NH, N]) -> [B, NH, stages]."""
    x = lf_stab[..., lo:lo + (hi - lo) // 8 * 8]
    return x.reshape(*x.shape[:-1], -1, 8).sum(-1)


# ---- CPU tests -----------------------------------------------------------------------------------------------------
def _coverage(name: str, DH: int = 64):
    sc = SCENARIOS[name]
    inp = make_inputs(sc, DH)
    m, lf, expb = gate_trace(inp)
    (a0, a1), (b0, b1) = calls(sc, 0)
    logF = torch.cat([stage_log_decay(lf, a0, a1), stage_log_decay(lf, b0, b1)], -1)
    return sc, inp, m, lf, expb, logF


@pytest.mark.parametrize("name", list(SCENARIOS))
def test_scenario_reaches_its_regime(name):
    sc, inp, m, lf, expb, logF = _coverage(name)
    below = (logF < LOG_MIN_DECAY).double().mean().item()
    under = int((lf < EXPF_UNDERFLOW).sum())
    exp_frac = expb.double().mean().item()
    print(f"{name}: stages F_8 < 1e-12 {below:.3f}, expf-underflow tokens {under}, exp(-m) denominator {exp_frac:.3f},"
          f" m in [{m.min():.1f}, {m.max():.1f}], stabilised log f >= {lf.min():.1f}")
    if name == "mild":
        assert below == 0 and lf.min() > -1.0 and -1.0 < m.min() and m.max() < 1.5
        assert 0.0 < exp_frac < 1.0
    elif name == "strong_forget":
        assert below > 0.85
        assert exp_frac > 0.5
    elif name == "straddle":
        assert 0.2 < below < 0.8
        per_head = (logF < LOG_MIN_DECAY).double().mean((0, 2))
        assert (per_head > 0.05).sum() >= 2 and (per_head < 0.95).sum() >= 2   # single heads cross the threshold
        assert (logF - LOG_MIN_DECAY).abs().min() < 0.05
    elif name == "spikes":
        big, _ = spike_positions(sc)
        assert under >= 2 * sc.B * len(big)
        hit = (lf < EXPF_UNDERFLOW).any(1).any(0)                 # positions where some (env, head) underflows
        for p in big:
            assert hit[p], f"no underflow at token {p}"
        assert below > 0.1 and lf.min() < -120
    elif name == "negative_m":
        assert m.max() < -25 and exp_frac == 1.0
    elif name == "long_memory":
        assert calls(sc, 0)[0][1] > 2048 and calls(sc, 1)[0][1] > 2048      # first calls span two super-chunks
        assert (m[..., 2047] - inp["m0"].double()).abs().min() > 2.0   # the super-chunk map moves m
        assert (logF > math.log(0.5)).double().mean() > 0.9
        assert m.max() - m.min() > 4.0


@pytest.mark.parametrize("name", list(SCENARIOS))
def test_fp32_oracle_meets_the_bound(name):
    """The plain fp32 oracle recurrence is within the GPU tests' bound of the float64 reference on every scenario."""
    sc = SCENARIOS[name]
    DH = 32
    inp = make_inputs(sc, DH)
    N = sc.base + TAIL
    ref = run_reference(inp, torch.float64, (sc.base, N))
    got = run_reference(inp, torch.float32, (sc.base, N))
    tol = BOUND + U_FP32 * ref["kappa"]
    (eh, rh), (eo, ro) = row_rel(got["h"], ref["h"], tol), row_rel(heads_rows(got["out"], sc.B, N),
                                                                    heads_rows(ref["out"], sc.B, N), tol)
    errs = dict(m=m_err(got["m"], ref["m"], ref["m_scale"]))
    for t in (sc.base, N):
        for j, part in enumerate("Cnm"):
            g, r = got["states"][t][j], ref["states"][t][j]
            errs[f"{part}@{t}"] = m_err(g, r, ref["m_scale"][..., t - 1]) if part == "m" else head_rel(g, r)
    print(name, f"h {eh:.2e} ({rh:.2f} of its bound) out {eo:.2e} ({ro:.2f})",
          " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert rh <= 1 and ro <= 1, (rh, ro)
    for k, e in errs.items():
        assert e <= (M_BOUND if k.startswith("m") else BOUND), (k, e)
    for x in (got["h"], got["out"]):
        assert torch.isfinite(x).all()



# ---- gate-heavy weights of the end-to-end tests ---------------------------------------------------------------------
# Per head of every mLSTM block: 0 strong forgetting (scenario 2), 1 input-gate spikes over strong forgetting
# (scenario 4), 2 m far below zero (scenario 5), 3 long memory. sLSTM blocks get the same per-head gate biases.
E2E_FGATE_B = (-4.0, -16.0, 1.0, 8.0)
E2E_IGATE_B = (0.0, -10.0, -30.0, 0.0)
E2E_SPIKE_GAIN = 11.5       # |w| / sqrt(3 inner) of head 1's input-gate row: pre-activations of std ~60, so that
                             # some spikes pass m by more than 104 (the cell inputs shrink as 1 / sqrt(width) here)


def gate_heavy_state_dict(cfg, seed: int = 0):
    """make_state_dict with a larger gate_std (input / forget pre-activations of std ~1.5 whatever the width), per-head
    igate / fgate bias overrides and head 1's input-gate weights scaled up (E2E_SPIKE_GAIN)."""
    from lram_b200.synth import make_state_dict
    sd = make_state_dict(cfg, seed=seed, gate_std=0.3 * math.sqrt(768.0 / (3 * cfg.inner)))
    for i in range(cfg.num_blocks):
        p = f"encoder.layers.blocks.{i}.xlstm."
        if cfg.is_slstm(i):
            b = sd[p + "slstm_cell._bias_"]                      # [NH, 4 (i, f, z, o), DHs]
            b[:, 0] = torch.tensor(E2E_IGATE_B).view(-1, 1)
            b[:, 1] = torch.tensor(E2E_FGATE_B).view(-1, 1)
            continue
        sd[p + "mlstm_cell.fgate.bias"] = torch.tensor(E2E_FGATE_B)
        sd[p + "mlstm_cell.igate.bias"] = torch.tensor(E2E_IGATE_B)
        w = sd[p + "mlstm_cell.igate.weight"]
        w[1] *= E2E_SPIKE_GAIN * math.sqrt(3 * cfg.inner) / w[1].norm()
    return sd


def oracle64(cfg, sd):
    """OracleEncoder with its weights recast to float64: fed float64 inputs it runs the whole stack in float64."""
    ora = O.OracleEncoder(cfg, sd)
    ora.sd = {k: v.double() for k, v in ora.sd.items()}
    return ora


def zero_state64(cfg, B: int):
    """The oracle's fresh state (what past_key_values=None means: zeros, m = 0) in float64: its sLSTM step would
    otherwise create float32 zeros and fail on float64 inputs."""
    z = dict(dtype=torch.float64)
    KS, NHc, DH = cfg.conv1d_kernel_size, cfg.num_heads, cfg.head_dim
    out = {}
    for i in range(cfg.num_blocks):
        if cfg.is_slstm(i):
            out[f"block_{i}"] = {"slstm_state": torch.zeros(4, B, cfg.d, **z),
                                 "conv_state": (torch.zeros(B, KS, cfg.d, **z),)}
        else:
            out[f"block_{i}"] = {"mlstm_state": (torch.zeros(B, NHc, DH, DH, **z), torch.zeros(B, NHc, DH, 1, **z),
                                                 torch.zeros(B, NHc, 1, 1, **z)),
                                 "conv_state": (torch.zeros(B, KS, cfg.inner, **z),)}
    return out


def run_oracle_recorded(ora, x, pkv=None):
    """ora.forward_cached(x, pkv) (pkv None: a fresh float64 state), recording for every mLSTM cell step the input gate, the stabilised log forget gate,
    m' and kappa (as run_reference) -> (hidden, state, rec) with rec[name] [tokens, mLSTM blocks, B, NH]."""
    cfg = ora.cfg
    nm = sum(not cfg.is_slstm(i) for i in range(cfg.num_blocks))
    step = O.recurrent_step_stabilized_simple
    calls_, absst, rec = [0], {}, {k: [] for k in ("ig", "lf", "m", "kappa", "ig_abs")}
    mblocks = [i for i in range(cfg.num_blocks) if not cfg.is_slstm(i)]

    def spy(c, n, m, q, k, v, ig, fg, eps=1e-6):
        blk = calls_[0] % nm
        calls_[0] += 1
        h, (c2, n2, m2) = step(c, n, m, q, k, v, ig, fg, eps)
        B, nh, _, DH = q.shape
        ca, na = absst.get(blk, (c.abs(), n.abs()))
        f, i = torch.exp(F.logsigmoid(fg) + m - m2), torch.exp(ig - m2)
        ka = k.abs().transpose(-1, -2) / math.sqrt(DH)
        ca = f * ca + i * (ka @ v.abs())
        na = f * na + i * ka
        absst[blk] = (ca, na)
        den = torch.maximum((q @ n2).abs(), torch.exp(-m2)) + eps
        num_max = (q @ c2).abs().amax(-1, keepdim=True).clamp_min(1e-300)
        kap = (q.abs() @ ca).amax(-1, keepdim=True) / num_max + (q.abs() @ na) / den
        # sum_j |w_j g_j| + |b| of the input-gate projection: its rounding reaches m wherever m' = i~
        gabs = torch.cat([t.reshape(B, nh * DH) for t in (q, k, v)], -1).abs()
        wi = ora._w(mblocks[blk], "xlstm.mlstm_cell.igate.weight").abs()
        ig_abs = gabs @ wi.t() + ora._w(mblocks[blk], "xlstm.mlstm_cell.igate.bias").abs()
        for name, val in (("ig", ig), ("lf", F.logsigmoid(fg) + m - m2), ("m", m2), ("kappa", kap), ("ig_abs", ig_abs)):
            rec[name].append(val.reshape(B, nh))
        return h, (c2, n2, m2)

    O.recurrent_step_stabilized_simple = spy
    try:
        y, st = ora.forward_cached(x, zero_state64(cfg, x.shape[0]) if pkv is None else pkv)
    finally:
        O.recurrent_step_stabilized_simple = step
    B, S = x.shape[:2]
    return y, st, {k: torch.stack(v).view(S, nm, B, NH) for k, v in rec.items()}


def assert_gate_heavy_coverage(rec, tag=""):
    """Every mLSTM block has a head in scenario 2 (stages with F_8 < 1e-12), 4 (expf underflow of the stabilised forget
    gate) and 5 (m far below zero) on the recorded gates; head 3 keeps a long memory. rec from run_oracle_recorded
    over >= 128 tokens (several records may be concatenated along the token axis)."""
    lf, m = rec["lf"], rec["m"]
    S = lf.shape[0] // 8 * 8
    for blk in range(lf.shape[1]):
        logF = lf[:S, blk].reshape(-1, 8, *lf.shape[2:]).sum(1)
        below = (logF < LOG_MIN_DECAY).double().mean((0, 1))
        under = (lf[:, blk] < EXPF_UNDERFLOW).sum((0, 1))
        print(f"{tag} block {blk}: stages F_8 < 1e-12 per head {[round(x, 2) for x in below.tolist()]}, "
              f"expf underflows {under.tolist()}, m min {[round(x, 1) for x in m[:, blk].amin((0, 1)).tolist()]}")
        assert below[0] > 0.6 and below[1] > 0.6 and below[3] == 0
        assert under[1] >= 2
        assert m[120:, blk, :, 2].max() < -25       # m falls from 0 by ~0.3 a token onto the input gate at -30


@pytest.mark.parametrize("name", ["toy128", "16M"])
def test_gate_heavy_weights_reach_the_regimes(name):
    """The end-to-end weights reach scenarios 2, 4 and 5 on the gates the float64 oracle records."""
    from lram_b200.config import preset
    cfg = preset(name, num_blocks=1)
    x = torch.randn(2, 200, cfg.d, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    y, _, rec = run_oracle_recorded(oracle64(cfg, gate_heavy_state_dict(cfg)), x)
    assert y.dtype == torch.float64
    assert_gate_heavy_coverage(rec, name)
