"""Generates the committed golden fixtures in this directory. Run in the BUILD container only:

    python tests/golden/make_golden.py

Sources of truth:
  tokenizer_kat.npz   — produced by the REFERENCE'S OWN code imported from the LRAM_REFERENCE_ROOT checkout
                        (`src/tokenizers_custom/{minmax,mu_law}_tokenizer.py`; they need only torch/numpy).
  hf_mlstm_step.npz   — produced by ``transformers.models.xlstm.modeling_xlstm.mlstm_recurrent_step_native``
                        (transformers 5.5.0 in this image): an independent implementation of the mLSTM
                        recurrent step by the xlstm authors. Convention differs (q scaled instead of k):
                        h equal, C_hf = sqrt(DH)*C, n_hf = sqrt(DH)*n.
  hf_mlstm_chunkwise.npz — ``mlstm_chunkwise_fw`` (48 tokens, chunk 16, non-zero initial (C, n, m)) and
                        ``xLSTMMultiHeadLayerNorm`` from the same transformers module.
  oracle_toy.npz      — produced by oracle/xlstm_oracle.py itself (regression pin + the vectors the GPU
                        parity tests re-check on the GPU, where no reference checkout is needed).

Nothing at test/bench time reads the reference checkout; only this script does.
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def _load_reference_tokenizers():
    import ref_stubs
    if not ref_stubs.reference_available():
        raise RuntimeError(ref_stubs.SKIP_REASON)
    base = os.path.join(ref_stubs.REFERENCE_ROOT, "src", "tokenizers_custom")
    pkg = types.ModuleType("ref_tok")
    pkg.__path__ = [base]
    sys.modules["ref_tok"] = pkg
    mods = {}
    for name in ("base_tokenizer", "minmax_tokenizer", "mu_law_tokenizer"):
        spec = importlib.util.spec_from_file_location(f"ref_tok.{name}", os.path.join(base, f"{name}.py"))
        m = importlib.util.module_from_spec(spec)
        sys.modules[f"ref_tok.{name}"] = m
        spec.loader.exec_module(m)
        mods[name] = m
    return mods


def make_tokenizer_kat():
    mods = _load_reference_tokenizers()
    MinMax = mods["minmax_tokenizer"].MinMaxTokenizer
    MinMax2 = mods["minmax_tokenizer"].MinMaxTokenizer2
    MuLaw = mods["mu_law_tokenizer"].MuLawTokenizer
    rng = np.random.default_rng(7)
    edge = np.array([-1.0, -0.999, 0.0, 0.5, 0.9999, 1.0, 1.5, -2.0, -0.9921875, 0.9921875,
                     1.0 - 2 ** -20, -1.0 + 2 ** -20, 0.0078125, -0.0078125, 0.00390625], dtype=np.float32)
    x = np.concatenate([edge, rng.uniform(-1.2, 1.2, size=4081).astype(np.float32)]).reshape(512, 8)
    xt = torch.from_numpy(x)
    out = {"x": x}
    for tag, tok in (("mm256s18", MinMax(vocab_size=256, shift=18)), ("mm64s0", MinMax(vocab_size=64, shift=0)),
                     ("mm100s0", MinMax(vocab_size=100, shift=0))):
        t = tok.tokenize(xt.clone())
        out[f"{tag}_tok"] = t.numpy().astype(np.int64)
        out[f"{tag}_inv"] = tok.inv_tokenize(t.clone()).numpy().astype(np.float32)
    # inverse over the whole id range the action head can emit (ids < shift decode to min_val)
    ids = torch.arange(0, 274, dtype=torch.long).view(1, -1)
    out["mm256s18_inv_all_ids"] = MinMax(vocab_size=256, shift=18).inv_tokenize(ids.clone()).numpy().astype(np.float32)
    tok2 = MinMax2(vocab_size=256, shift=18)
    t2 = tok2.tokenize(xt.clone())
    out["mm2_256s18_tok"] = t2.numpy().astype(np.int64)
    out["mm2_256s18_inv"] = tok2.inv_tokenize(t2.clone()).numpy().astype(np.float32)
    mu = MuLaw(vocab_size=256, shift=0)
    xc = xt.clamp(-1, 1)
    tm = mu.tokenize(xc.clone())
    out["mulaw_x"] = xc.numpy()
    out["mulaw256_tok"] = tm.numpy().astype(np.int64)
    out["mulaw256_inv"] = mu.inv_tokenize(tm.clone()).numpy().astype(np.float32)
    np.savez_compressed(os.path.join(HERE, "tokenizer_kat.npz"), **out)
    print("tokenizer_kat.npz", {k: v.shape for k, v in out.items()})


def make_hf_step():
    from transformers.models.xlstm import modeling_xlstm as hf
    step = hf.mlstm_recurrent_step_native
    g = torch.Generator().manual_seed(11)
    B, NH, DH, T = 2, 4, 32, 12
    q = torch.randn(T, B, NH, DH, generator=g)
    k = torch.randn(T, B, NH, DH, generator=g)
    v = torch.randn(T, B, NH, DH, generator=g)
    ig = torch.randn(T, B, NH, 1, generator=g) * 2.0
    fg = torch.randn(T, B, NH, 1, generator=g) * 2.0 + 2.0
    c = torch.zeros(B, NH, DH, DH)
    n = torch.zeros(B, NH, DH)
    m = torch.zeros(B, NH, 1)
    hs = []
    for t in range(T):
        h, (c, n, m) = step(q[t], k[t], v[t], ig[t], fg[t], c, n, m, eps=1e-6)
        hs.append(h)
    out = dict(q=q.numpy(), k=k.numpy(), v=v.numpy(), ig=ig.numpy(), fg=fg.numpy(),
               h=torch.stack(hs).numpy(), c_final=c.numpy(), n_final=n.numpy(), m_final=m.numpy())
    np.savez_compressed(os.path.join(HERE, "hf_mlstm_step.npz"), **out)
    print("hf_mlstm_step.npz", {k_: v_.shape for k_, v_ in out.items()})


def make_hf_chunkwise_and_norm():
    """Two more vectors from transformers' xlstm code (same authors as the pip `xlstm` the reference calls):
    the chunkwise-parallel forward over a sequence STARTING FROM A NON-ZERO STATE (pins the recurrence across many
    steps and the state hand-over the prefill relies on) and the multi-head LayerNorm (pins the GroupNorm form)."""
    from transformers.models.xlstm import modeling_xlstm as hf
    g = torch.Generator().manual_seed(23)
    B, NH, DH, S = 2, 4, 32, 48
    q = torch.randn(B, NH, S, DH, generator=g)
    k = torch.randn(B, NH, S, DH, generator=g)
    v = torch.randn(B, NH, S, DH, generator=g)
    ig = torch.randn(B, NH, S, generator=g) * 2.0
    fg = torch.randn(B, NH, S, generator=g) * 2.0 + 2.0
    c0 = torch.randn(B, NH, DH, DH, generator=g) * 0.3
    n0 = torch.randn(B, NH, DH, generator=g) * 0.3
    m0 = torch.randn(B, NH, 1, generator=g)
    # transformers 5.5.0 writes `fgate.logsigmoid(vecF)` (no such Tensor method): give it the obvious meaning for
    # the duration of the call; every other line executed is transformers' own
    torch.Tensor.logsigmoid = lambda self, x: torch.nn.functional.logsigmoid(x)
    try:
        H, _, _, last, _ = hf.mlstm_chunkwise_fw(q, k, v, ig, fg, cstate=c0, nstate=n0, mstate=m0,
                                                 return_last_states=True, chunk_size=16, eps=1e-6)
    finally:
        del torch.Tensor.logsigmoid
    out = dict(q=q.numpy(), k=k.numpy(), v=v.numpy(), ig=ig.numpy(), fg=fg.numpy(), c0=c0.numpy(), n0=n0.numpy(),
               m0=m0.numpy(), h=H.numpy(), c_final=last[0].numpy(), n_final=last[1].numpy(), m_final=last[2].numpy())
    ln = hf.xLSTMMultiHeadLayerNorm(num_heads=NH, head_dim=DH, eps=1e-5, use_weight=True, use_bias=False)
    w_res = torch.randn(NH * DH, generator=g) * 0.1          # xlstm 1.0.x stores the residual: gamma = 1 + w
    with torch.no_grad():
        ln.weight.copy_(1.0 + w_res)
        x = torch.randn(B, 5, NH, DH, generator=g) * 3.0 + 0.5
        y = ln(x)
    out.update(ln_x=x.numpy(), ln_w_residual=w_res.numpy(), ln_y=y.numpy())
    np.savez_compressed(os.path.join(HERE, "hf_mlstm_chunkwise.npz"), **out)
    print("hf_mlstm_chunkwise.npz", {k_: v_.shape for k_, v_ in out.items()})


def make_oracle_toy():
    from lram_b200.config import preset
    from lram_b200.synth import make_state_dict, make_stream
    from oracle.xlstm_oracle import OraclePolicy
    out = {}
    for name, B, steps in (("toy", 5, 6), ("toy128", 3, 4)):
        cfg = preset(name)
        sd = make_state_dict(cfg, seed=0)
        pol = OraclePolicy(cfg, sd)
        states, rtg, _ = make_stream(cfg, range(B), steps, domains="mixed", seed=1234)
        pkv = None
        toks, hids, acts = [], [], []
        for t in range(steps):
            o = pol.step(torch.from_numpy(states[t]), torch.from_numpy(rtg[t]), past_key_values=pkv)
            pkv = o["past_key_values"]
            toks.append(o["action_tokens"].numpy())
            acts.append(o["action_preds"].numpy())
            hids.append(o["last_hidden_state"].numpy())
        out[f"{name}_states"] = states
        out[f"{name}_rtg"] = rtg
        out[f"{name}_tokens"] = np.stack(toks).astype(np.int64)
        out[f"{name}_actions"] = np.stack(acts).astype(np.float32)
        out[f"{name}_hidden"] = np.stack(hids).astype(np.float32)
        last = pkv[f"block_{cfg.num_blocks - 1}"]
        out[f"{name}_C_last"] = last["mlstm_state"][0].numpy()
        out[f"{name}_n_last"] = last["mlstm_state"][1].numpy()
        out[f"{name}_m_last"] = last["mlstm_state"][2].numpy()
        out[f"{name}_conv_last"] = last["conv_state"][0].numpy()
    np.savez_compressed(os.path.join(HERE, "oracle_toy.npz"), **out)
    print("oracle_toy.npz", {k_: v_.shape for k_, v_ in out.items()})


if __name__ == "__main__":
    torch.manual_seed(0)
    torch.set_num_threads(1)
    make_tokenizer_kat()
    make_hf_step()
    make_hf_chunkwise_and_norm()
    make_oracle_toy()
