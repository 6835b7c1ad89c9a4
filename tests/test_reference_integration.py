"""The encoder swap, exercised against the REAL reference classes (needs a reference checkout: LRAM_REFERENCE_ROOT).

What is real here: the reference's `MultiDomainDiscreteDecisionXLSTMModel` (constructed by its own `__init__`), its
`load_state_dict`, its `forward` / `compute_hidden_states` / `handle_inference_cache` / `get_predictions`, its agent's
`predict`, its `custom_evaluate_policy` — imported unmodified through tests/golden/ref_stubs.py. What is swapped in is
`policy.encoder = FusedXLSTMEncoder(config=policy.config)`, the one-line edit INTEGRATION.md §2 describes for
`src/algos/models/decision_xlstm.py:188-189`.

The reference checkout and a GPU need not be on the same machine, so the CUDA engine does not run in this
test: `XLSTMEngine` is replaced BY THE TEST with a double (`_OracleEngine`, below) that answers `encoder_step` with the
CPU oracle. The product has no such path (its engine raises without CUDA — asserted below); what this test proves is
the host-side contract: parameter names / shapes / load order, lazy engine build after `load_state_dict`, the `forward`
signature, and every way the reference reads the returned object. The same `FusedXLSTMEncoder` code runs with the real
engine in tests/test_ref_golden.py::test_cuda_encoder_swap_equals_reference_hidden on the GPU.
"""
import os
import sys
import warnings

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import ref_stubs  # noqa: E402

from lram_b200 import decision_xlstm as DX  # noqa: E402
from lram_b200.config import preset  # noqa: E402
from lram_b200.engine import StateCache  # noqa: E402
from lram_b200.image_encoder import make_impala_state_dict  # noqa: E402
from lram_b200.synth import make_state_dict  # noqa: E402

needs_reference = pytest.mark.skipif(not ref_stubs.reference_available(), reason=ref_stubs.SKIP_REASON)


class _OracleCache(StateCache):
    def __init__(self, engine, B):            # no device buffer: the double keeps the oracle's dict
        self.engine, self.B, self.pkv = engine, B, None


class _OracleEngine:
    """Test double for XLSTMEngine(encoder_only=True): same constructor and methods, CPU oracle inside."""
    built = 0

    def __init__(self, cfg, state_dict, max_batch, device=None, encoder_only=False):
        from oracle.xlstm_oracle import OracleEncoder
        assert encoder_only, "the encoder swap must build an encoder-only engine"
        need = {f"encoder.layers.blocks.{i}.xlstm.proj_up.weight" for i in range(cfg.num_blocks)}
        assert need <= set(state_dict), "engine built before the weights were loaded"
        self.cfg, self.max_batch, self.device, self.encoder_only = cfg, max_batch, torch.device("cpu"), True
        self.enc = OracleEncoder(cfg, state_dict)
        self.closed = False
        type(self).built += 1

    def new_state(self, B):
        return _OracleCache(self, B)

    def encoder_step(self, cache, x, mode=0, flags=0, out=None):
        hs, cache.pkv = self.enc.forward_cached(x, cache.pkv)
        if out is not None:
            out.copy_(hs)
            return out
        return hs

    def close(self):
        self.closed = True


@pytest.fixture()
def ref():
    ref_stubs.install()
    import make_ref_golden as G
    return G


def test_product_engine_refuses_to_run_without_cuda():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    cfg = preset("toy")
    enc = DX.FusedXLSTMEncoder(config=cfg)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        enc(inputs_embeds=torch.zeros(1, 3, cfg.d), use_cache=True)


@needs_reference
def test_swap_then_load_state_dict_then_reference_rollout(ref, monkeypatch, golden_dir):
    tag = "toy128_metaworld"
    z = np.load(os.path.join(golden_dir, "ref_rollout.npz"))
    seed, n_episodes, ep_len = (int(v) for v in z[f"{tag}.meta"])
    target_return, reward_scale = (float(v) for v in z[f"{tag}.scalars"])
    cfg = preset("toy128")
    sd = make_state_dict(cfg, seed=seed)
    sd.update(make_impala_state_dict(cfg.d, ref.IMAGE_SHAPE, seed=seed + 100))

    # 1. the reference builds its policy with its own (random) init; nothing of ours is loaded yet
    import gym
    from src.algos.models.decision_xlstm import MultiDomainDiscreteDecisionXLSTMModel, xLSTMEncoder
    blank = {k: torch.zeros_like(v) for k, v in sd.items()}
    policy = ref.build_reference_policy(cfg, blank)
    assert isinstance(policy.encoder, xLSTMEncoder)
    ref_keys = {k for k in policy.state_dict() if k.startswith("encoder.")}

    # 2. the swap of decision_xlstm.py:188-189, with the policy's own xLSTMConfig
    monkeypatch.setattr(DX, "XLSTMEngine", _OracleEngine)
    _OracleEngine.built = 0
    del policy.encoder
    policy.encoder = DX.FusedXLSTMEncoder(config=policy.config)
    policy.encoder.reset_parameters()                         # what post_init() calls (decision_xlstm.py:211-214)
    assert {k for k in policy.state_dict() if k.startswith("encoder.")} == ref_keys      # same names as xlstm's
    assert _OracleEngine.built == 0                                                      # nothing built yet

    # 3. the reference's loader runs AFTER construction (decision_transformer_sb3.py:1120-1184)
    res = policy.load_state_dict(sd, strict=False)
    assert not [k for k in res.missing_keys if k.startswith("encoder.")]
    assert not res.unexpected_keys
    for k in ref_keys:
        assert torch.equal(policy.state_dict()[k], sd[k]), k
    assert _OracleEngine.built == 0

    # 4. the reference's own rollout loop + agent.predict through the swapped encoder
    from src.callbacks.evaluation import custom_evaluate_policy
    obs = z[f"{tag}.obs"]
    env = ref_stubs.ScriptedVecEnv(obs, gym.spaces.Box(-1, 1, (4,), np.float32),
                                   gym.spaces.Box(-1, 1, (39,), np.float32), ep_len=ep_len)
    agent = ref.build_reference_agent(policy, cfg, target_return / reward_scale, reward_scale)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _, ep_lengths, _ = custom_evaluate_policy(agent, env, n_eval_episodes=n_episodes, return_episode_rewards=True)
    got = np.stack([np.asarray(a).reshape(-1) for a in env.actions_seen])
    assert np.array_equal(got, z[f"{tag}.actions"])           # identical to the run with the reference's own encoder
    assert [int(v) for v in ep_lengths] == [int(v) for v in z[f"{tag}.ep_lengths"]]
    assert _OracleEngine.built == 1                           # one lazy build, reused over resets and episodes

    # 5. loading other weights invalidates the engine; the next call rebuilds it from the new parameters
    first = policy.encoder._engine
    policy.load_state_dict(make_state_dict(cfg, seed=seed + 1), strict=False)
    assert first.closed and policy.encoder._engine is None
    out = policy.encoder(inputs_embeds=torch.zeros(2, 3, cfg.d), use_cache=True)
    assert _OracleEngine.built == 2 and out["last_hidden_state"].shape == (2, 3, cfg.d)
    assert out.get("past_key_values") is not None and out.hidden_states is None and out.attentions is None


@needs_reference
def test_whole_policy_mirror_loads_a_reference_checkpoint(ref):
    """`policy.state_dict()` of the REFERENCE model (every key it has, incl. the ones the path never reads) loads into
    our `MultiDomainDiscreteDecisionXLSTMModel` built with the reference's constructor signature."""
    cfg = preset("toy128")
    sd = make_state_dict(cfg, seed=3)
    sd.update(make_impala_state_dict(cfg.d, ref.IMAGE_SHAPE, seed=103))
    policy = ref.build_reference_policy(cfg, sd)
    ckpt = {"module._orig_mod." + k: v for k, v in policy.state_dict().items()}     # DDP + torch.compile prefixes
    assert any(k.endswith("embed_timestep.weight") for k in ckpt)
    import gym
    ours = DX.MultiDomainDiscreteDecisionXLSTMModel.from_reference_args(
        policy.config, gym.spaces.Box(0, 255, ref.IMAGE_SHAPE, dtype=np.uint8), gym.spaces.Discrete(15),
        stochastic_policy=False, reward_condition=True, tokenize_a=True, tokenize_rtg=False, action_channels=256,
        discrete_actions=18, state_dim=204, image_shape=[3, 64, 64], relative_pos_embds=False, use_time_embds=False,
        action_condition=False, shared_a_head=True, max_act_dim=8)
    ours.load_state_dict(ckpt)
    mine = ours.state_dict()
    for k, v in policy.state_dict().items():
        if k in mine:
            assert torch.equal(mine[k], v), k
    hot = [k for k in mine if not k.startswith("embed_image.")]
    assert set(hot) <= set(policy.state_dict())
    assert ours.cfg.d == cfg.d and ours.cfg.num_blocks == cfg.num_blocks and ours.cfg.act_dim == 8
    with pytest.raises(NotImplementedError):
        DX.MultiDomainDiscreteDecisionXLSTMModel.from_reference_args(policy.config, None, None, action_condition=True)
    bad = dict(ckpt)
    bad.pop("module._orig_mod.embed_ln.bias")
    with pytest.raises(KeyError, match="embed_ln.bias"):
        ours.load_state_dict(bad)


@needs_reference
def test_action_sampling_equals_reference_sample_from_logits(ref):
    """`a_sample_kwargs` (discrete_decision_transformer_sb3.py:62-63): our restatement draws the reference's samples
    under the same torch seed, for the shapes the reference can sample ([1, 274] discrete head, [274] per-dimension)."""
    from src.algos.models.model_utils import sample_from_logits as ref_sample
    g = torch.Generator().manual_seed(3)
    for shape in ((1, 274), (274,)):
        logits = torch.randn(*shape, generator=g) * 3
        for kw in (dict(temperature=1.0, top_k=0, top_p=0.5), dict(temperature=0.7, top_k=5, top_p=0.0),
                   dict(temperature=1.3, top_k=0, top_p=0.9)):
            for seed in range(5):
                torch.manual_seed(seed)
                a = ref_sample(logits.clone(), **kw)
                torch.manual_seed(seed)
                b = DX.sample_from_logits(logits.clone(), **kw)
                assert torch.equal(a, b), (shape, kw, seed)


# ---- without the reference: the same two restatements, pinned by their documented behaviour --------------------------
def test_policy_from_reference_args_loads_a_prefixed_checkpoint():
    """`from_reference_args` with a reference-style config (HF fields + `xlstm_config` dict) builds the toy128 policy;
    a DDP + torch.compile prefixed checkpoint carrying off-path keys loads into it, and a missing hot-path key raises."""
    import types
    cfg = preset("toy128")
    conf = types.SimpleNamespace(hidden_size=cfg.d, n_layer=cfg.num_blocks, xlstm_config={
        "embedding_dim": cfg.d, "num_blocks": cfg.num_blocks,
        "mlstm_block": {"mlstm": {"num_heads": cfg.num_heads, "conv1d_kernel_size": cfg.conv1d_kernel_size,
                                  "qkv_proj_blocksize": cfg.qkv_proj_blocksize}}})
    ours = DX.MultiDomainDiscreteDecisionXLSTMModel.from_reference_args(
        conf, None, None, stochastic_policy=False, reward_condition=True, tokenize_a=True, tokenize_rtg=False,
        action_channels=256, discrete_actions=18, state_dim=204, image_shape=[3, 64, 64], relative_pos_embds=False,
        use_time_embds=False, action_condition=False, shared_a_head=True, max_act_dim=8)
    assert (ours.cfg.d, ours.cfg.num_blocks, ours.cfg.num_heads, ours.cfg.act_dim) == (cfg.d, cfg.num_blocks, 4, 8)
    sd = make_state_dict(cfg, seed=3)
    sd.update(make_impala_state_dict(cfg.d, (3, 64, 64), seed=103))
    sd.update({"embed_timestep.weight": torch.ones(16, cfg.d), "predict_state.weight": torch.ones(204, cfg.d)})
    ckpt = {"module._orig_mod." + k: v for k, v in sd.items()}
    ours.load_state_dict(ckpt)
    mine = ours.state_dict()
    assert set(mine) <= set(sd) and "embed_timestep.weight" not in mine
    for k, v in mine.items():
        assert torch.equal(v, sd[k]), k
    with pytest.raises(NotImplementedError):
        DX.MultiDomainDiscreteDecisionXLSTMModel.from_reference_args(conf, None, None, action_condition=True)
    bad = dict(ckpt)
    bad.pop("module._orig_mod.embed_ln.bias")
    with pytest.raises(KeyError, match="embed_ln.bias"):
        ours.load_state_dict(bad)


def test_action_sampling_keeps_only_the_allowed_tokens():
    """`sample_from_logits`: draws stay inside the top-k set and above the top_p quantile, repeat under the same torch
    seed, keep the reference's shapes, and `temperature` multiplies the logits (a large one concentrates on the max)."""
    g = torch.Generator().manual_seed(3)
    for shape in ((1, 274), (274,)):
        logits = torch.randn(*shape, generator=g) * 3
        top5 = set(torch.topk(logits.reshape(-1), 5).indices.tolist())
        cut = torch.quantile(logits.double().reshape(-1), 0.5).item()
        for seed in range(20):
            torch.manual_seed(seed)
            a = DX.sample_from_logits(logits.clone(), temperature=1.0, top_k=5, top_p=0.0)
            assert a.shape == shape[:-1] and int(a.reshape(-1)[0]) in top5
            b = DX.sample_from_logits(logits.clone(), temperature=1.0, top_k=0, top_p=0.5)
            assert logits.reshape(-1)[int(b.reshape(-1)[0])].item() > cut
            torch.manual_seed(seed)
            assert torch.equal(DX.sample_from_logits(logits.clone(), temperature=1.0, top_k=5, top_p=0.0), a)
            hot = DX.sample_from_logits(logits.clone(), temperature=1e4, top_k=0, top_p=0.9)
            assert int(hot.reshape(-1)[0]) == int(logits.reshape(-1).argmax())
