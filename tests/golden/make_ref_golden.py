"""Golden vectors produced by the REFERENCE'S OWN hot-path code. Run in the BUILD container only:

    python tests/golden/make_ref_golden.py

What runs (unmodified, imported from the LRAM_REFERENCE_ROOT checkout through tests/golden/ref_stubs.py):
  * `MultiDomainDiscreteDecisionXLSTMModel.__init__` / `.forward(use_inference_cache=True)`
    (src/algos/models/decision_xlstm.py:175-289, online_decision_transformer_model.py:326-530,588-612,
    discrete_decision_transformer_model.py:236-383, multi_domain_discrete_dt_model.py:12-108),
  * `xLSTMEncoder.forward` (decision_xlstm.py:138-169) and the reference's `load_state_dict`,
  * `DiscreteDecisionXLSTM.predict / pad_inputs / get_action_pred`
    (src/algos/decision_xlstm.py:11-35, decision_transformer_sb3.py:621-667, discrete_decision_transformer_sb3.py:13-72),
  * `custom_evaluate_policy` (src/callbacks/evaluation.py:14-271) on a scripted one-env VecEnv,
  * the reference's tokenizers (src/tokenizers_custom).
What does NOT come from the reference: the third-party `xlstm` package (absent) is the stand-in `oracle/xlstm_shim.py`
(the oracle's arithmetic under xlstm's module / parameter names). These vectors therefore pin the LRAM-side logic —
embedding, token interleave, embed_ln, cache trimming, output slicing, head, argmax, inv_tokenize, padding, rollout
bookkeeping — for the oracle AND for the CUDA path; the cell arithmetic keeps its `transformers` pins.

Weights: `lram_b200.synth.make_state_dict(cfg, seed)` loaded into the reference model with ITS `load_state_dict`
(strict=False; the keys it leaves at their init are asserted to be off the hot path). Tests rebuild the same weights from
the seed, so the fixtures hold inputs' seeds and outputs only.

Files written (tests/golden/): ref_policy_forward/<case>.npz (one file per case keeps each under 1 MB), ref_rollout.npz
"""
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import ref_stubs  # noqa: E402

from lram_b200.config import preset  # noqa: E402
from lram_b200.image_encoder import make_impala_state_dict  # noqa: E402
from lram_b200.synth import make_state_dict, make_stream  # noqa: E402

IMAGE_SHAPE = (3, 64, 64)
C_STRIDE = (37, 41)
# keys of the reference model that the hot path never reads (asserted when loading the synthetic weights)
OFF_PATH_PREFIXES = ("embed_timestep.", "embed_action.", "predict_state.", "predict_return.", "predict_reward.",
                     "predict_action.", "embed_image.", "embed_action_disc.")


def build_reference_policy(cfg, sd, with_image: bool = True):
    """The reference's own policy object for `cfg`, carrying the synthetic weights `sd`."""
    ref_stubs.install()
    import gym
    from src.algos.models.decision_xlstm import MultiDomainDiscreteDecisionXLSTMModel, xLSTMConfig
    xl = {"mlstm_block": {"mlstm": {"conv1d_kernel_size": cfg.conv1d_kernel_size,
                                    "qkv_proj_blocksize": cfg.qkv_proj_blocksize, "num_heads": cfg.num_heads}},
          "slstm_block": {"slstm": {"backend": "cuda", "num_heads": cfg.num_heads,
                                    "conv1d_kernel_size": cfg.conv1d_kernel_size,
                                    "bias_init": "powerlaw_blockdependent"},
                          "feedforward": {"proj_factor": cfg.ffn_proj_factor, "act_fn": "gelu"}},
          "context_length": 150, "num_blocks": cfg.num_blocks, "embedding_dim": cfg.d}
    if cfg.slstm_at:
        xl["slstm_at"] = list(cfg.slstm_at)
    # configs/agent_params/huggingface/xlstm_*.yaml + builder.py:56-60
    hf = xLSTMConfig(state_dim=cfg.state_dim, act_dim=cfg.act_dim, max_ep_len=1000, max_length=50,
                     n_layer=cfg.num_blocks, hidden_size=cfg.d, n_head=cfg.num_heads, xlstm_config=xl)
    # train env of the multi-domain runs is Procgen bigfish: image observations, Discrete(15) (SURVEY.md §8)
    obs_space = gym.spaces.Box(0, 255, IMAGE_SHAPE, dtype=np.uint8)
    act_space = gym.spaces.Discrete(15)
    # configs/agent_params/model_kwargs/multi_domain.yaml:1-11 + builder.py:63-65 (max_act_dim)
    policy = MultiDomainDiscreteDecisionXLSTMModel(
        hf, obs_space, act_space, stochastic_policy=False, reward_condition=True, tokenize_a=True, tokenize_rtg=False,
        action_channels=cfg.action_channels, discrete_actions=cfg.discrete_actions, state_dim=cfg.state_dim,
        image_shape=list(IMAGE_SHAPE), relative_pos_embds=False, use_time_embds=False, action_condition=False,
        shared_a_head=True, max_act_dim=cfg.act_dim)
    res = policy.load_state_dict(sd, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    left = [k for k in res.missing_keys if not k.startswith(OFF_PATH_PREFIXES)]
    assert not left, f"hot-path keys not covered by the synthetic state_dict: {left}"
    if with_image:
        assert not [k for k in res.missing_keys if k.startswith("embed_image.")]
    return policy.eval()


def build_reference_agent(policy, cfg, target_return: float, reward_scale: float):
    """The reference's agent class with the attributes `predict` and the rollout loop read, without running SB3's
    `OffPolicyAlgorithm.__init__` (training set-up, out of scope)."""
    from src.algos.decision_xlstm import DiscreteDecisionXLSTM

    class _Buf:
        max_state_dim, max_act_dim, seqs_per_sample = cfg.state_dim, cfg.act_dim, 1

        def __len__(self):
            return 0

    agent = object.__new__(DiscreteDecisionXLSTM)
    agent.__dict__.update(
        policy=policy, device=torch.device("cpu"), use_inference_cache=True, past_key_values=None,
        replay_buffer=_Buf(), s_proj_raw=False, s_proj_dim=None, a_proj_dim=None, transforms=None, state_mean=None,
        state_std=None, reset_inf_cache_freq=None, ddp_kwargs={}, use_amp=False, amp_dtype=torch.bfloat16,
        target_return_type="fixed", target_return=target_return, _reward_scale=reward_scale, a_sample_kwargs=None,
        rtg_sample_kwargs={}, eval_context_len=5, persist_context=False, compile=False, _last_target_return=None,
        num_timesteps=0, log_attn_maps=False)
    return agent


def _np(t):
    return t.detach().cpu().numpy()


@torch.no_grad()
def policy_forward_case(out, tag, cfg_name, seed, B, n_steps, discrete, image=False, domains="mixed"):
    """Batched `policy.forward` with a carried cache, growing histories exactly as the rollout loop feeds them."""
    cfg = preset(cfg_name)
    sd = make_state_dict(cfg, seed=seed)
    sd.update(make_impala_state_dict(cfg.d, IMAGE_SHAPE, seed=seed + 100))
    policy = build_reference_policy(cfg, sd)
    states_np, rtg_np, _ = make_stream(cfg, range(B), n_steps, domains=domains, seed=4321)
    rng = np.random.default_rng(99)
    frames = rng.integers(0, 256, (n_steps, B) + IMAGE_SHAPE, dtype=np.uint8) if image else None
    act_dim = 1 if discrete else cfg.act_dim
    pkv = None
    rec = {k: [] for k in ("action_preds", "action_logits", "last_hidden_state", "tokens")}
    for t in range(n_steps):
        lo = max(0, t - 3)                                      # the loop keeps <= 4 timesteps (evaluation.py:172-177)
        if image:
            states = torch.from_numpy(frames[lo:t + 1]).transpose(0, 1).float()          # [B,T,C,H,W] raw 0..255 floats
        else:
            states = torch.from_numpy(states_np[lo:t + 1]).transpose(0, 1).contiguous()  # [B,T,204]
        T = states.shape[1]
        rtg = torch.from_numpy(rtg_np[lo:t + 1]).transpose(0, 1).reshape(B, T, 1)
        actions = torch.zeros(B, T, act_dim)                                             # evaluation.py:131
        rewards = torch.zeros(B, T, 1)                                                   # evaluation.py:132
        timesteps = torch.arange(lo, t + 1).repeat(B, 1)
        mask = torch.ones(B, T, dtype=torch.long)
        o = policy(states=states, actions=actions, rewards=rewards, returns_to_go=rtg, timesteps=timesteps,
                   attention_mask=mask, return_dict=True, deterministic=True, prompt=None, task_id=None,
                   ddp_kwargs={}, use_inference_cache=True, past_key_values=pkv)
        pkv = o.past_key_values
        rec["action_preds"].append(_np(o.action_preds))
        rec["action_logits"].append(_np(o.action_logits))
        rec["last_hidden_state"].append(_np(o.last_hidden_state))
        # `last_encoder_output` [B, 3, 1, d] is last_hidden_state reshaped/permuted (online...model.py:453-459)
        assert torch.equal(o.last_encoder_output[:, :, 0], o.last_hidden_state)
        lg = o.action_logits
        rec["tokens"].append(_np(torch.argmax(lg[..., :cfg.discrete_actions] if discrete else lg, dim=-1)))
    for k, v in rec.items():
        out[f"{tag}.{k}"] = np.stack(v)
    # final recurrent state of block 0 and the last block (C, n, m, conv) — the reference's past_key_values dict
    for bi in (0, cfg.num_blocks - 1):
        st = pkv[f"block_{bi}"]
        if "mlstm_state" in st:
            c, n, m = st["mlstm_state"]
            # C of the big presets is stored as a strided sample (C_STRIDE rows x columns) to keep the fixture small
            out[f"{tag}.block{bi}.C"] = _np(c if c.numel() <= 300_000 else c[:, :, ::C_STRIDE[0], ::C_STRIDE[1]])
            out[f"{tag}.block{bi}.n"], out[f"{tag}.block{bi}.m"] = _np(n), _np(m)
        out[f"{tag}.block{bi}.conv"] = _np(st["conv_state"][0])
    out[f"{tag}.meta"] = np.array([seed, B, n_steps, int(discrete), int(image)], dtype=np.int64)
    out[f"{tag}.cfg"] = np.array(cfg_name)
    out[f"{tag}.domains"] = np.array(domains)
    if image:
        out[f"{tag}.frames"] = frames
    print(tag, {k: out[f"{tag}.{k}"].shape for k in rec})


@torch.no_grad()
def rollout_case(out, tag, cfg_name, seed, kind, n_episodes, ep_len, persist_context=False, reset_inf_cache_freq=None):
    """`custom_evaluate_policy` + `DiscreteDecisionXLSTM.predict`, one env, scripted observations."""
    ref_stubs.install()
    import gym
    from src.callbacks.evaluation import custom_evaluate_policy
    cfg = preset(cfg_name)
    sd = make_state_dict(cfg, seed=seed)
    sd.update(make_impala_state_dict(cfg.d, IMAGE_SHAPE, seed=seed + 100))
    policy = build_reference_policy(cfg, sd)
    n_obs = n_episodes * ep_len + 1
    rng = np.random.default_rng(seed + 7)
    if kind == "metaworld":            # Box(39) observations, Box(4) actions: continuous branch, padded 39->204, 4->8
        obs = rng.uniform(-1, 1, (n_obs, 39)).astype(np.float32)
        obs_space, act_space = gym.spaces.Box(-1, 1, (39,), np.float32), gym.spaces.Box(-1, 1, (4,), np.float32)
        target_return, reward_scale = 100.0, 200.0
    elif kind == "atari":              # uint8 frames, Discrete(18): discrete branch through embed_image
        obs = rng.integers(0, 256, (n_obs,) + IMAGE_SHAPE, dtype=np.uint8)
        obs_space, act_space = gym.spaces.Box(0, 255, IMAGE_SHAPE, np.uint8), gym.spaces.Discrete(18)
        target_return, reward_scale = 90.0, 1.0
    else:
        raise ValueError(kind)
    env = ref_stubs.ScriptedVecEnv(obs, act_space, obs_space, ep_len=ep_len)
    agent = build_reference_agent(policy, cfg, target_return / reward_scale, reward_scale)
    agent.persist_context = persist_context                  # evaluation.py:213-237: context carried over episode ends
    agent.reset_inf_cache_freq = reset_inf_cache_freq        # decision_transformer_sb3.py:663-666
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ep_rewards, ep_lengths, _ = custom_evaluate_policy(agent, env, n_eval_episodes=n_episodes,
                                                           return_episode_rewards=True)
    out[f"{tag}.obs"] = obs
    out[f"{tag}.actions"] = np.stack([np.asarray(a).reshape(-1) for a in env.actions_seen])
    out[f"{tag}.ep_lengths"] = np.array(ep_lengths, dtype=np.int64)
    out[f"{tag}.meta"] = np.array([seed, n_episodes, ep_len], dtype=np.int64)
    out[f"{tag}.flags"] = np.array([int(persist_context), -1 if reset_inf_cache_freq is None else reset_inf_cache_freq],
                                   dtype=np.int64)
    out[f"{tag}.scalars"] = np.array([target_return, reward_scale], dtype=np.float64)
    out[f"{tag}.cfg"] = np.array(cfg_name)
    out[f"{tag}.kind"] = np.array(kind)
    print(tag, out[f"{tag}.actions"].shape, out[f"{tag}.actions"][:2], ep_lengths)


def main():
    torch.manual_seed(0)
    torch.set_num_threads(max(1, (os.cpu_count() or 2) // 2))
    fwd = {}
    policy_forward_case(fwd, "toy128_cont", "toy128", seed=11, B=5, n_steps=6, discrete=False)
    policy_forward_case(fwd, "toy128_disc", "toy128", seed=12, B=5, n_steps=6, discrete=True)
    policy_forward_case(fwd, "toy128_img_disc", "toy128", seed=13, B=2, n_steps=3, discrete=True, image=True)
    policy_forward_case(fwd, "toy128ms_cont", "toy128-ms", seed=14, B=3, n_steps=4, discrete=False)
    policy_forward_case(fwd, "16M_cont", "16M", seed=15, B=2, n_steps=4, discrete=False, domains="dmcontrol")
    policy_forward_case(fwd, "48M_cont", "48M", seed=16, B=2, n_steps=3, discrete=False, domains="metaworld")
    policy_forward_case(fwd, "110M_disc", "110M", seed=17, B=2, n_steps=3, discrete=True, domains="mixed")
    policy_forward_case(fwd, "206M_cont", "206M", seed=18, B=1, n_steps=2, discrete=False, domains="mimicgen")
    os.makedirs(os.path.join(HERE, "ref_policy_forward"), exist_ok=True)
    for tag in dict.fromkeys(k.split(".")[0] for k in fwd):
        f = os.path.join(HERE, "ref_policy_forward", f"{tag}.npz")
        np.savez_compressed(f, **{k: v for k, v in fwd.items() if k.split(".")[0] == tag})
        print(os.path.relpath(f, HERE), os.path.getsize(f), "bytes")
    ro = {}
    rollout_case(ro, "toy128_metaworld", "toy128", seed=21, kind="metaworld", n_episodes=3, ep_len=7)
    rollout_case(ro, "toy128_atari", "toy128", seed=22, kind="atari", n_episodes=2, ep_len=5)
    rollout_case(ro, "16M_metaworld", "16M", seed=23, kind="metaworld", n_episodes=2, ep_len=6)
    rollout_case(ro, "toy128_persist", "toy128", seed=24, kind="metaworld", n_episodes=3, ep_len=5, persist_context=True)
    rollout_case(ro, "toy128_resetfreq", "toy128", seed=25, kind="metaworld", n_episodes=2, ep_len=9,
                 reset_inf_cache_freq=4)
    np.savez_compressed(os.path.join(HERE, "ref_rollout.npz"), **ro)
    print("ref_rollout.npz", os.path.getsize(os.path.join(HERE, "ref_rollout.npz")), "bytes")


if __name__ == "__main__":
    main()
