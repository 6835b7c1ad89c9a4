"""Parity against vectors produced by the REFERENCE'S OWN model / agent / rollout code
(tests/golden/ref_policy_forward/<case>.npz, ref_rollout.npz; generator tests/golden/make_ref_golden.py runs the
reference's `MultiDomainDiscreteDecisionXLSTMModel.forward`, `DiscreteDecisionXLSTM.predict` and
`custom_evaluate_policy` through stub packages, with the absent `xlstm` package stood in by oracle/xlstm_shim.py).

CPU (`-m "not gpu"`): the oracle's LRAM-side restatement (embed, token layout, cache trim, head slice, argmax,
inv_tokenize, rollout bookkeeping) == the reference's code; and, when LRAM_REFERENCE_ROOT points at a checkout of the
reference, the fixtures regenerate bit-identically from it.
GPU (`-m gpu`): the CUDA path through the host mirror == the reference's outputs: action tokens / argmax actions
bit-exact, hidden states / logits / recurrent state within REL_TOL = 1e-3 (north_star's tolerance).
"""
import os
import sys

import numpy as np
import pytest
import torch

from lram_b200.config import preset
from lram_b200.image_encoder import make_impala_state_dict
from lram_b200.synth import make_state_dict, make_stream

REL_TOL = 1e-3
IMAGE_SHAPE = (3, 64, 64)
C_STRIDE = (37, 41)
FWD_TAGS = ["toy128_cont", "toy128_disc", "toy128_img_disc", "toy128ms_cont", "16M_cont", "48M_cont", "110M_disc",
            "206M_cont"]
# persist: `persist_context` (evaluation.py:213-237) — the recurrent state survives episode ends;
# resetfreq: `reset_inf_cache_freq` (decision_transformer_sb3.py:663-666) — the cache is dropped every 4 timesteps
ROLLOUT_TAGS = ["toy128_metaworld", "toy128_atari", "16M_metaworld", "toy128_persist", "toy128_resetfreq"]
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def fwd(golden_dir):
    d = os.path.join(golden_dir, "ref_policy_forward")
    out = {}
    for tag in FWD_TAGS:
        with np.load(os.path.join(d, f"{tag}.npz")) as z:
            out.update({k: z[k] for k in z.files})
    return out


@pytest.fixture(scope="module")
def rollouts(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_rollout.npz"))


def _case(z, tag):
    seed, B, n_steps, discrete, image = (int(v) for v in z[f"{tag}.meta"])
    cfg = preset(str(z[f"{tag}.cfg"]))
    sd = make_state_dict(cfg, seed=seed)
    sd.update(make_impala_state_dict(cfg.d, IMAGE_SHAPE, seed=seed + 100))
    states_np, rtg_np, _ = make_stream(cfg, range(B), n_steps, domains=str(z[f"{tag}.domains"]), seed=4321)
    frames = z[f"{tag}.frames"] if image else None
    return cfg, sd, B, n_steps, bool(discrete), states_np, rtg_np, frames


def _rel(a, b):
    a, b = torch.as_tensor(a, dtype=torch.float64), torch.as_tensor(b, dtype=torch.float64)
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _sample_c(c):
    return c if c.numel() <= 300_000 else c[:, :, ::C_STRIDE[0], ::C_STRIDE[1]]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: oracle == reference
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", FWD_TAGS)
def test_oracle_policy_equals_reference_forward(fwd, tag):
    from oracle.xlstm_oracle import OraclePolicy
    cfg, sd, B, n_steps, discrete, states_np, rtg_np, frames = _case(fwd, tag)
    if cfg.d >= 768 and os.environ.get("LRAM_FAST_TESTS"):
        pytest.skip("large preset skipped in fast mode")
    ora = OraclePolicy(cfg, sd)
    pkv = None
    for t in range(n_steps):
        s = torch.from_numpy(frames[t]) if frames is not None else torch.from_numpy(states_np[t])
        o = ora.step(s, torch.from_numpy(rtg_np[t]), past_key_values=pkv, discrete=discrete)
        pkv = o["past_key_values"]
        assert np.array_equal(o["action_tokens"].numpy().reshape(B, -1), fwd[f"{tag}.tokens"][t].reshape(B, -1)), t
        assert np.array_equal(o["action_preds"].numpy().reshape(B, -1),
                              fwd[f"{tag}.action_preds"][t].reshape(B, -1)), t
        assert _rel(o["last_hidden_state"], fwd[f"{tag}.last_hidden_state"][t]) < 1e-5
        assert _rel(o["action_logits"].reshape(B, -1), fwd[f"{tag}.action_logits"][t].reshape(B, -1)) < 1e-5
    for bi in (0, cfg.num_blocks - 1):
        st = pkv[f"block_{bi}"]
        if "mlstm_state" in st:
            c, n, m = st["mlstm_state"]
            assert _rel(_sample_c(c), fwd[f"{tag}.block{bi}.C"]) < 1e-5
            assert _rel(n, fwd[f"{tag}.block{bi}.n"]) < 1e-5 and _rel(m, fwd[f"{tag}.block{bi}.m"]) < 1e-5
        assert _rel(st["conv_state"][0], fwd[f"{tag}.block{bi}.conv"]) < 1e-5


def _oracle_rollout(z, tag):
    """The oracle policy driven by the reference loop's bookkeeping (rtg update, reset on done), one env."""
    from oracle.xlstm_oracle import OraclePolicy
    seed, n_episodes, ep_len = (int(v) for v in z[f"{tag}.meta"])
    target_return, reward_scale = (float(v) for v in z[f"{tag}.scalars"])
    cfg = preset(str(z[f"{tag}.cfg"]))
    kind = str(z[f"{tag}.kind"])
    sd = make_state_dict(cfg, seed=seed)
    sd.update(make_impala_state_dict(cfg.d, IMAGE_SHAPE, seed=seed + 100))
    ora = OraclePolicy(cfg, sd)
    obs = z[f"{tag}.obs"]
    persist, freq = (int(v) for v in z[f"{tag}.flags"]) if f"{tag}.flags" in z.files else (0, -1)
    target = np.float32(target_return / reward_scale)
    rtg, pkv, acts = target, None, []
    for k in range(n_episodes * ep_len):
        o = obs[k]
        if kind == "atari":
            s = torch.from_numpy(o)[None]
            out = ora.step(s, torch.tensor([rtg]), past_key_values=pkv, discrete=True)
            acts.append(out["action_preds"].numpy().reshape(-1)[:1].astype(np.int64))
        else:
            s = torch.zeros(1, cfg.state_dim)
            s[0, : o.shape[0]] = torch.from_numpy(o)
            out = ora.step(s, torch.tensor([rtg]), past_key_values=pkv, discrete=False)
            acts.append(out["action_preds"].numpy().reshape(-1)[:4])
        pkv = out["past_key_values"]
        ts = k % ep_len                                  # timestep of the prediction just made
        if freq > 0 and ts > 0 and ts % freq == 0:
            pkv = None                                   # reset_inf_cache_freq
        if (k + 1) % ep_len == 0:
            rtg = target
            if not persist:
                pkv = None
        else:
            rtg = np.float32(rtg - np.float32(1.0) / np.float32(reward_scale))
    return np.stack(acts)


@pytest.mark.parametrize("tag", ROLLOUT_TAGS)
def test_oracle_rollout_equals_reference_rollout(rollouts, tag):
    acts = _oracle_rollout(rollouts, tag)
    ref = rollouts[f"{tag}.actions"]
    assert acts.shape == ref.shape
    assert np.array_equal(acts.astype(ref.dtype), ref)
    seed, n_episodes, ep_len = (int(v) for v in rollouts[f"{tag}.meta"])
    assert list(rollouts[f"{tag}.ep_lengths"]) == [ep_len * (i + 1) for i in range(n_episodes)]   # :209 (sic): cumulative


def _ref_stubs():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import ref_stubs
    return ref_stubs


def test_fixtures_regenerate_from_the_reference(fwd, rollouts):
    """Only with a checkout of the reference (LRAM_REFERENCE_ROOT): the committed fixtures are what the reference's own
    code produces today."""
    ref_stubs = _ref_stubs()
    if not ref_stubs.reference_available():
        pytest.skip(ref_stubs.SKIP_REASON)
    import make_ref_golden as G
    out = {}
    G.policy_forward_case(out, "toy128_cont", "toy128", seed=11, B=5, n_steps=6, discrete=False)
    G.policy_forward_case(out, "toy128_disc", "toy128", seed=12, B=5, n_steps=6, discrete=True)
    for k, v in out.items():
        if v.dtype.kind in "iu":
            assert np.array_equal(v, fwd[k]), k
        elif v.dtype.kind == "f" and not k.endswith("action_preds"):
            assert _rel(v, fwd[k]) < 1e-5, k                # BLAS thread count may differ from the generating run
        elif v.dtype.kind == "f":
            assert np.array_equal(v, fwd[k]), k             # decoded actions: exact (they are functions of the tokens)
    ro = {}
    G.rollout_case(ro, "toy128_atari", "toy128", seed=22, kind="atari", n_episodes=2, ep_len=5)
    assert np.array_equal(ro["toy128_atari.actions"], rollouts["toy128_atari.actions"])


# ---------------------------------------------------------------------------------------------------------------------
# GPU: CUDA path == reference
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("use_graph", [False, True])
@pytest.mark.parametrize("tag", FWD_TAGS)
def test_cuda_policy_equals_reference_forward(fwd, tag, use_graph):
    """Our `MultiDomainDiscreteDecisionXLSTMModel.forward`, fed the same growing histories the reference was fed."""
    from lram_b200.decision_xlstm import MultiDomainDiscreteDecisionXLSTMModel
    cfg, sd, B, n_steps, discrete, states_np, rtg_np, frames = _case(fwd, tag)
    if frames is None:
        sd = {k: v for k, v in sd.items() if not k.startswith("embed_image.")}
    policy = MultiDomainDiscreteDecisionXLSTMModel(cfg, sd, max_batch=B, use_graph=use_graph)
    pkv = None
    act_dim = 1 if discrete else cfg.act_dim
    for t in range(n_steps):
        lo = max(0, t - 3)
        if frames is not None:
            states = torch.from_numpy(frames[lo:t + 1]).transpose(0, 1).float()        # raw 0..255 as floats
        else:
            states = torch.from_numpy(states_np[lo:t + 1]).transpose(0, 1).contiguous()
        T = states.shape[1]
        rtg = torch.from_numpy(rtg_np[lo:t + 1]).transpose(0, 1).reshape(B, T, 1)
        o = policy(states=states, actions=torch.zeros(B, T, act_dim), rewards=torch.zeros(B, T, 1), returns_to_go=rtg,
                   timesteps=torch.arange(lo, t + 1).repeat(B, 1), attention_mask=torch.ones(B, T, dtype=torch.long),
                   return_dict=True, use_inference_cache=True, past_key_values=pkv)
        pkv = o.past_key_values
        ref_tok = fwd[f"{tag}.tokens"][t].reshape(B, -1)
        got_tok = o.action_tokens.cpu().numpy().reshape(B, -1)[:, : ref_tok.shape[1]]
        assert np.array_equal(got_tok, ref_tok), (t, got_tok, ref_tok)
        assert np.array_equal(o.action_preds.cpu().numpy().reshape(B, -1),
                              fwd[f"{tag}.action_preds"][t].reshape(B, -1)), t
        assert tuple(o.action_preds.shape) == fwd[f"{tag}.action_preds"][t].shape
        assert tuple(o.action_logits.shape) == fwd[f"{tag}.action_logits"][t].shape
        assert _rel(o.last_hidden_state.cpu(), fwd[f"{tag}.last_hidden_state"][t]) < REL_TOL
        assert _rel(o.action_logits.cpu(), fwd[f"{tag}.action_logits"][t]) < REL_TOL
    ref_pkv = pkv.to_past_key_values()
    for bi in (0, cfg.num_blocks - 1):
        st = ref_pkv[f"block_{bi}"]
        if "mlstm_state" in st:
            c, n, m = (x.cpu() for x in st["mlstm_state"])
            assert _rel(_sample_c(c), fwd[f"{tag}.block{bi}.C"]) < REL_TOL
            assert _rel(n, fwd[f"{tag}.block{bi}.n"]) < REL_TOL and _rel(m, fwd[f"{tag}.block{bi}.m"]) < REL_TOL
        assert _rel(st["conv_state"][0].cpu(), fwd[f"{tag}.block{bi}.conv"]) < REL_TOL


@gpu
@pytest.mark.parametrize("use_graph", [True, False])
@pytest.mark.parametrize("tag", ["toy128_cont", "16M_cont", "toy128ms_cont"])
def test_cuda_encoder_swap_equals_reference_hidden(fwd, tag, use_graph):
    """Encoder-only integration (the swap at decision_xlstm.py:188-189): an `nn.Module` `FusedXLSTMEncoder(config=...)`
    whose `layers.*` parameters are filled by `load_state_dict` AFTER construction, engine built lazily; embeddings by
    the checker (oracle). last_hidden_state must equal what the reference's encoder produced inside its policy."""
    from lram_b200.decision_xlstm import FusedXLSTMEncoder
    from oracle.xlstm_oracle import OraclePolicy
    cfg, sd, B, n_steps, discrete, states_np, rtg_np, _ = _case(fwd, tag)
    enc = FusedXLSTMEncoder(config=cfg, max_batch=B, use_graph=use_graph)
    enc_sd = {k[len("encoder."):]: v for k, v in sd.items() if k.startswith("encoder.")}
    res = enc.load_state_dict(enc_sd)
    assert not res.missing_keys and not res.unexpected_keys
    ora = OraclePolicy(cfg, sd)
    pkv = None
    for t in range(n_steps):
        x = ora.embed(torch.from_numpy(states_np[t]), torch.from_numpy(rtg_np[t]), torch.zeros(B))
        out = enc(inputs_embeds=x.cuda(), past_key_values=pkv, use_cache=True)
        pkv = out.get("past_key_values")
        assert _rel(out["last_hidden_state"].cpu(), fwd[f"{tag}.last_hidden_state"][t]) < REL_TOL
    assert enc.engine.encoder_only


@gpu
@pytest.mark.parametrize("tag", ROLLOUT_TAGS)
def test_cuda_rollout_equals_reference_rollout(rollouts, tag):
    """`lram_b200.rollout.custom_evaluate_policy` (reference signature) with our agent on the scripted env the reference
    loop ran on: the actions the env receives must be bit-identical, the episode accounting equal."""
    from lram_b200.decision_xlstm import DiscreteDecisionXLSTM, MultiDomainDiscreteDecisionXLSTMModel
    from lram_b200.rollout import custom_evaluate_policy
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from ref_stubs import Box, Discrete, ScriptedVecEnv
    z = rollouts
    seed, n_episodes, ep_len = (int(v) for v in z[f"{tag}.meta"])
    target_return, reward_scale = (float(v) for v in z[f"{tag}.scalars"])
    cfg = preset(str(z[f"{tag}.cfg"]))
    kind = str(z[f"{tag}.kind"])
    sd = make_state_dict(cfg, seed=seed)
    sd.update(make_impala_state_dict(cfg.d, IMAGE_SHAPE, seed=seed + 100))
    persist, freq = (int(v) for v in z[f"{tag}.flags"]) if f"{tag}.flags" in z.files else (0, -1)
    policy = MultiDomainDiscreteDecisionXLSTMModel(cfg, sd, max_batch=1)
    agent = DiscreteDecisionXLSTM(policy, target_return=target_return / reward_scale, reward_scale=reward_scale,
                                  persist_context=bool(persist), reset_inf_cache_freq=freq if freq > 0 else None)
    if kind == "atari":
        spaces = (Discrete(18), Box(0, 255, IMAGE_SHAPE, np.uint8))
    else:
        spaces = (Box(-1, 1, (4,), np.float32), Box(-1, 1, (39,), np.float32))
    env = ScriptedVecEnv(z[f"{tag}.obs"], spaces[0], spaces[1], ep_len=ep_len)
    ep_rewards, ep_lengths, ep_times = custom_evaluate_policy(agent, env, n_eval_episodes=n_episodes,
                                                               return_episode_rewards=True, warn=False)
    got = np.stack([np.asarray(a).reshape(-1) for a in env.actions_seen])
    ref = z[f"{tag}.actions"]
    assert got.shape == ref.shape and np.array_equal(got.astype(ref.dtype), ref)
    assert [int(v) for v in ep_lengths] == [int(v) for v in z[f"{tag}.ep_lengths"]]
    assert len(ep_rewards) == n_episodes and len(ep_times) == n_episodes
    assert agent.past_key_values is None


@gpu
def test_cuda_batched_rollout_equals_single_env_rollouts():
    """num_envs = 3 through the batched loop == three independent one-env runs (envs never interact), with episode ends
    at different steps per env, and `persist_context` keeping the recurrent state over episode ends."""
    from lram_b200.decision_xlstm import DiscreteDecisionXLSTM, MultiDomainDiscreteDecisionXLSTMModel
    from lram_b200.rollout import custom_evaluate_policy
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from ref_stubs import Box
    cfg = preset("toy128")
    sd = make_state_dict(cfg, seed=5)
    policy = MultiDomainDiscreteDecisionXLSTMModel(cfg, sd, max_batch=3)
    rng = np.random.default_rng(3)
    obs = rng.uniform(-1, 1, (3, 40, 39)).astype(np.float32)
    ep_lens = (4, 6, 5)

    class VecEnv:
        def __init__(self, ids):
            self.ids, self.num_envs = list(ids), len(ids)
            self.action_space, self.observation_space = Box(-1, 1, (4,), np.float32), Box(-1, 1, (39,), np.float32)
            self.cur, self.t, self.seen = [0] * len(ids), [0] * len(ids), [[] for _ in ids]

        def _o(self, k):
            o = obs[self.ids[k], self.cur[k]]
            self.cur[k] += 1
            return o

        def reset(self):
            return np.stack([self._o(k) for k in range(self.num_envs)])

        def step(self, actions):
            actions = np.asarray(actions).reshape(self.num_envs, -1)
            done = np.zeros(self.num_envs, dtype=bool)
            for k in range(self.num_envs):
                self.seen[k].append(actions[k].copy())
                self.t[k] += 1
                if self.t[k] >= ep_lens[self.ids[k]]:
                    done[k], self.t[k] = True, 0
            return (np.stack([self._o(k) for k in range(self.num_envs)]), np.ones(self.num_envs, np.float32), done,
                    [{} for _ in range(self.num_envs)])

    for persist in (False, True):
        agent = DiscreteDecisionXLSTM(policy, target_return=0.5, reward_scale=200.0, persist_context=persist)
        batched = VecEnv([0, 1, 2])
        custom_evaluate_policy(agent, batched, n_eval_episodes=6, warn=False)
        for i in range(3):
            single = VecEnv([i])
            custom_evaluate_policy(agent, single, n_eval_episodes=2, warn=False)
            n = len(single.seen[0])
            assert n == 2 * ep_lens[i]
            assert np.array_equal(np.stack(single.seen[0]), np.stack(batched.seen[i][:n])), (persist, i)
