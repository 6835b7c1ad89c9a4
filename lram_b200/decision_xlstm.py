"""Host-side mirror of the reference's operator / plugin interface for the hot path.

  FusedXLSTMEncoder                      <->  xLSTMEncoder                         src/algos/models/decision_xlstm.py:119-172
  MultiDomainDiscreteDecisionXLSTMModel  <->  same name                            src/algos/models/decision_xlstm.py:281-289
                                              (.forward: online_decision_transformer_model.py:326-390)
  DiscreteDecisionXLSTM (agent)          <->  same name (predict / pad_inputs / get_action_pred)
                                              src/algos/decision_xlstm.py:6-35, decision_transformer_sb3.py:621-667,
                                              discrete_decision_transformer_sb3.py:13-72

Both model classes are `nn.Module`s that own their weights as parameters under the REFERENCE'S state-dict names
(`encoder.layers.blocks.{i}.xlstm.proj_up.weight`, `embed_state.weight`, `action_net.0.weight`, ...), so the
reference's order of operations works unchanged: construct (`del self.encoder; self.encoder = ...`,
decision_xlstm.py:188-189) -> `load_state_dict` (decision_transformer_sb3.py:1120-1184) -> `.to(device)` -> call.
The CUDA engine (C-ABI handle + packed bf16/fp32 device copies of the weights) is built LAZILY on the first call and
rebuilt after every `load_state_dict` / `reset_parameters`.

Same names, argument meaning and error behaviour as the reference for this path; everything that is not on
the inference-cache rollout path (training, losses, prompts, autoregressive per-dimension decoding) is out of
scope and raises NotImplementedError instead of silently doing something else. Image observations run the
reference's ImpalaCNN in PyTorch/cuDNN (image_encoder.py) and enter the CUDA path as state embeddings.
All arithmetic runs in libxlstm_b200.so; there is no PyTorch fallback.
"""
from __future__ import annotations

import dataclasses
import math
import weakref
from typing import Any, Dict, Optional

import torch
import torch.nn as nn

from . import _lib as L
from .config import XLSTMPolicyConfig
from .engine import StateCache, XLSTMEngine, strip_checkpoint_prefixes
from .image_encoder import ImpalaCNN, embed_frames, scale_frames
from .tokenizers import make_tokenizer


class _Output(dict):
    """dict with attribute access, like HF ModelOutput: supports out['k'], out.k, out.get('k')."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            return None


class _Tree(nn.Module):
    """Parameter container; nested so that `state_dict()` yields the reference's dotted names."""


def _add_param(root: nn.Module, dotted: str, shape, value: float = 0.0) -> None:
    parts = dotted.split(".")
    mod = root
    for p in parts[:-1]:
        if not hasattr(mod, p):
            mod.add_module(p, _Tree())
        mod = getattr(mod, p)
    mod.register_parameter(parts[-1], nn.Parameter(torch.full(tuple(shape), float(value)), requires_grad=False))


def encoder_param_shapes(cfg: XLSTMPolicyConfig) -> Dict[str, tuple]:
    """name (relative to `encoder.`) -> shape, for every tensor of the xlstm block stack (SURVEY.md Appendix A)."""
    d, inner, NH, KS, bs = cfg.d, cfg.inner, cfg.num_heads, cfg.conv1d_kernel_size, cfg.qkv_proj_blocksize
    out: Dict[str, tuple] = {}
    for i in range(cfg.num_blocks):
        p = f"layers.blocks.{i}."
        out[p + "xlstm_norm.weight"] = (d,)
        if cfg.is_slstm(i):
            dh, ff = d // NH, cfg.ffn_dim
            out[p + "xlstm.conv1d.conv.weight"] = (d, 1, KS)
            out[p + "xlstm.conv1d.conv.bias"] = (d,)
            for g in ("fgate", "igate", "zgate", "ogate"):
                out[p + f"xlstm.{g}.weight"] = (NH, dh, dh)
            out[p + "xlstm.slstm_cell._recurrent_kernel_"] = (NH, dh, 4, dh)
            out[p + "xlstm.slstm_cell._bias_"] = (NH, 4, dh)
            out[p + "xlstm.group_norm.weight"] = (d,)
            out[p + "ffn_norm.weight"] = (d,)
            out[p + "ffn.proj_up.weight"] = (2 * ff, d)
            out[p + "ffn.proj_down.weight"] = (d, ff)
            continue
        out[p + "xlstm.proj_up.weight"] = (2 * inner, d)
        for g in ("q_proj", "k_proj", "v_proj"):
            out[p + f"xlstm.{g}.weight"] = (inner // bs, bs, bs)
        out[p + "xlstm.conv1d.conv.weight"] = (inner, 1, KS)
        out[p + "xlstm.conv1d.conv.bias"] = (inner,)
        out[p + "xlstm.mlstm_cell.igate.weight"] = (NH, 3 * inner)
        out[p + "xlstm.mlstm_cell.igate.bias"] = (NH,)
        out[p + "xlstm.mlstm_cell.fgate.weight"] = (NH, 3 * inner)
        out[p + "xlstm.mlstm_cell.fgate.bias"] = (NH,)
        out[p + "xlstm.mlstm_cell.outnorm.weight"] = (inner,)
        out[p + "xlstm.learnable_skip"] = (inner,)
        out[p + "xlstm.proj_down.weight"] = (d, inner)
    out["layers.post_blocks_norm.weight"] = (d,)
    return out


def config_from_reference(hf_config, **policy_kwargs) -> XLSTMPolicyConfig:
    """`xLSTMConfig` (decision_xlstm.py:104-116: HF DecisionTransformerConfig + `xlstm_config` dict laid out as
    configs/agent_params/huggingface/xlstm_*.yaml:7-26) -> XLSTMPolicyConfig. Unsupported options raise."""
    if isinstance(hf_config, XLSTMPolicyConfig):
        return dataclasses.replace(hf_config, **policy_kwargs) if policy_kwargs else hf_config
    xl = hf_config.xlstm_config
    xl = dict(xl) if not isinstance(xl, dict) else xl
    if getattr(hf_config, "ln_bias", False) or getattr(hf_config, "rms_norm", False):
        raise NotImplementedError("ln_bias / rms_norm variants are off in every shipped preset and not implemented")
    if getattr(hf_config, "chunkwise_step", False):
        raise NotImplementedError("chunkwise_step is an unimplemented-upstream hook (decision_xlstm.py:158-159)")
    m = dict(dict(xl.get("mlstm_block") or {}).get("mlstm") or {})
    kw = dict(embedding_dim=int(xl.get("embedding_dim", getattr(hf_config, "hidden_size", 0))),
              num_blocks=int(xl.get("num_blocks", getattr(hf_config, "n_layer", 0))),
              num_heads=int(m.get("num_heads", 4)), conv1d_kernel_size=int(m.get("conv1d_kernel_size", 4)),
              qkv_proj_blocksize=int(m.get("qkv_proj_blocksize", 4)), proj_factor=float(m.get("proj_factor", 2.0)),
              slstm_at=tuple(int(i) for i in (xl.get("slstm_at") or ())))
    if kw["slstm_at"]:
        ff = dict(dict(xl.get("slstm_block") or {}).get("feedforward") or {})
        kw["ffn_proj_factor"] = float(ff.get("proj_factor", 1.3))
    for k in ("state_dim", "act_dim"):
        if getattr(hf_config, k, None) is not None:
            kw[k] = int(getattr(hf_config, k))
    kw.update(policy_kwargs)
    cfg = XLSTMPolicyConfig(name="reference", **kw)
    cfg.validate()
    return cfg


class FusedXLSTMEncoder(nn.Module):
    """Drop-in for `xLSTMEncoder` on the `use_cache=True` path: `forward(inputs_embeds=..., past_key_values=...,
    use_cache=True)` returns `last_hidden_state` [B, n_tok, d] and the (opaque) `past_key_values`. With
    `use_cache=False` it returns the hidden states of every token from a zero state and `past_key_values=None` (the
    reference's non-cache branch; `past_key_values` is not read there). Inputs that require grad with grad enabled raise
    NotImplementedError: there is no training path.

    Construct it like the reference constructs its encoder, `FusedXLSTMEncoder(config=config)` with the policy's
    `xLSTMConfig` (or an `XLSTMPolicyConfig`): the parameters `layers.blocks.{i}....` / `layers.post_blocks_norm.weight`
    are registered immediately, so the policy's `load_state_dict` fills them; the engine is built on the first forward
    from whatever the parameters hold then. (`FusedXLSTMEncoder(engine)` wraps an existing engine instead.)

    The reference treats `past_key_values` opaquely (only `is None` tests, SURVEY.md §8 a13); here it is a
    `StateCache` living on the GPU and updated IN PLACE (the returned object is the one passed in).
    A reference-format dict ({"block_i": {...}}) is accepted too and imported into a fresh cache.
    """

    def __init__(self, config=None, mode: int = L.XL_MODE_PER_TOKEN, max_batch: int = 64, device=None,
                 use_graph: bool = True, **_unused):
        super().__init__()
        self.use_graph = use_graph        # replay the step from a CUDA graph (persistent input / output staging buffers)
        self._io: Dict[tuple, tuple] = {}
        self._engine: Optional[XLSTMEngine] = None
        self._owns_engine = True
        self._engine_provider = None      # set by a policy that shares its (full) engine with this encoder
        self.mode = mode
        self.max_batch = int(max_batch)
        self._device = torch.device(device) if device is not None else None
        if isinstance(config, XLSTMEngine):                      # wrap an engine somebody else built (a policy's)
            self._engine, self._owns_engine = config, False
            self.cfg = config.cfg
            self.max_batch = config.max_batch
        else:
            if config is None:
                raise ValueError("FusedXLSTMEncoder needs the policy's xLSTMConfig (or an XLSTMPolicyConfig / engine)")
            self.cfg = config_from_reference(config)
            for name, shape in encoder_param_shapes(self.cfg).items():
                _add_param(self, name, shape)
            self.reset_parameters()
            self.register_load_state_dict_post_hook(lambda module, incompatible: module.invalidate_engine())
        self.config = self.cfg

    # ---- weights ---------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def reset_parameters(self):
        """`post_init` hook of the reference (decision_xlstm.py:211-214) -> xLSTMBlockStack.reset_parameters():
        norms weight 0 (gamma = 1 + w), skip 1, gate weights 0, fgate bias linspace(3, 6), igate bias N(0, 0.1),
        proj_up / q,k,v small-init, proj_down wang-init (SURVEY.md Appendix A)."""
        if not self._owns_engine:
            return None
        cfg = self.cfg
        small = math.sqrt(2.0 / (5.0 * cfg.d))
        wang = 2.0 / (cfg.num_blocks * math.sqrt(cfg.d))
        ks_bound = 1.0 / math.sqrt(cfg.conv1d_kernel_size)
        for name, p in self.named_parameters():
            if name.endswith(("xlstm_norm.weight", "ffn_norm.weight", "post_blocks_norm.weight", "outnorm.weight",
                              "group_norm.weight", "mlstm_cell.igate.weight", "mlstm_cell.fgate.weight")):
                p.zero_()
            elif name.endswith("learnable_skip"):
                p.fill_(1.0)
            elif name.endswith("mlstm_cell.fgate.bias"):
                p.copy_(torch.linspace(3.0, 6.0, p.numel()))
            elif name.endswith("mlstm_cell.igate.bias"):
                p.normal_(0.0, 0.1)
            elif name.endswith("proj_down.weight"):
                p.normal_(0.0, wang)
            elif name.endswith(("conv.weight", "conv.bias")):
                p.uniform_(-ks_bound, ks_bound)
            elif name.endswith("_bias_"):
                p.zero_()
                p[:, 1, :] = torch.linspace(3.0, 6.0, p.shape[-1])
            else:                                   # proj_up, headwise q/k/v and sLSTM gates, recurrent kernel
                p.normal_(0.0, small)
        self.invalidate_engine()
        return None

    def invalidate_engine(self):
        self._io.clear()
        if self._owns_engine and self._engine is not None:
            self._engine.close()
            self._engine = None

    def _build_engine(self) -> XLSTMEngine:
        sd = {"encoder." + k: v for k, v in self.state_dict().items()}
        dev = self._device
        if dev is None:
            p = next(self.parameters())
            dev = p.device if p.is_cuda else torch.device("cuda", torch.cuda.current_device()) \
                if torch.cuda.is_available() else p.device
        return XLSTMEngine(self.cfg, sd, max_batch=self.max_batch, device=dev, encoder_only=True)

    @property
    def engine(self) -> XLSTMEngine:
        if self._engine_provider is not None:
            return self._engine_provider()
        if self._engine is None:
            self._engine = self._build_engine()
        return self._engine

    # ---- xLSTMEncoder.forward (decision_xlstm.py:138-169) -----------------------------------------------------------
    def forward(self, input_ids=None, past_key_values=None, attention_mask=None, token_type_ids=None,
                position_ids=None, head_mask=None, inputs_embeds=None, encoder_hidden_states=None,
                encoder_attention_mask=None, use_cache=None, output_attentions=None, output_hidden_states=None,
                return_dict=None):
        if inputs_embeds is None:
            raise ValueError("xLSTM encoder consumes already embedded inputs (inputs_embeds)")
        if not use_cache and torch.is_grad_enabled() and inputs_embeds.requires_grad:
            raise NotImplementedError("training (autograd through the encoder) is out of scope of the inference path")
        engine = self.engine
        B = inputs_embeds.shape[0]
        if B > engine.max_batch and self._owns_engine and self._engine_provider is None:   # grow the workspace
            self.max_batch = B
            self.invalidate_engine()
            engine = self.engine
        if not use_cache:
            # the non-cache branch (decision_xlstm.py:166-167, xLSTMBlockStack.forward(x)): every token from a zero
            # state, no cache kept or read; computed by the chunkwise prefill, which equals the parallel form
            hs = engine.prefill(engine.new_state(B), inputs_embeds.detach().to(engine.device, torch.float32))
            return _Output(last_hidden_state=hs, past_key_values=None, hidden_states=None, attentions=None)
        if past_key_values is None:
            cache = engine.new_state(B)                        # zeros == state None (m starts at 0)
        elif isinstance(past_key_values, StateCache):
            cache = past_key_values
            if cache.engine is not engine:                     # engine rebuilt (weights reloaded): same layout
                cache.engine = engine
        elif isinstance(past_key_values, dict):
            cache = engine.new_state(B)
            cache.load_past_key_values(past_key_values)
        else:
            raise TypeError(f"unsupported past_key_values type {type(past_key_values)}")
        if cache.B != B:
            raise ValueError(f"past_key_values holds {cache.B} envs, inputs have batch {B}")
        x = inputs_embeds.detach().to(engine.device, torch.float32)
        if x.shape[1] > 4:
            # a whole context at once: what `chunkwise_step` (decision_xlstm.py:158-159) asks of layers.step
            hs = engine.prefill(cache, x)
        elif self.use_graph:
            # a graph is keyed on its pointers: stage the step's input / output in persistent buffers
            key = (id(engine), B, x.shape[1])
            io = self._io.get(key)
            if io is None:
                io = (torch.empty_like(x, memory_format=torch.contiguous_format), torch.empty_like(x))
                self._io[key] = io
            io[0].copy_(x, non_blocking=True)
            engine.encoder_step(cache, io[0], mode=self.mode, flags=L.XL_FLAG_GRAPH, out=io[1])
            hs = io[1].clone()
        else:
            hs = engine.encoder_step(cache, x, mode=self.mode)
        return _Output(last_hidden_state=hs, past_key_values=cache, hidden_states=None, attentions=None)


_POLICY_HOT_KEYS = ("embed_state.weight", "embed_state.bias", "embed_return.weight", "embed_return.bias",
                    "embed_rewards.weight", "embed_rewards.bias", "embed_ln.weight", "embed_ln.bias",
                    "action_net.0.weight", "action_net.0.bias")
# tensors of a reference checkpoint that exist but are never read on this path (SURVEY.md App. C.3, C.9)
_OFF_PATH_PREFIXES = ("embed_timestep.", "embed_action.", "embed_action_disc.", "predict_state.", "predict_return.",
                      "predict_reward.", "predict_action.", "embed_act_pos.")


class MultiDomainDiscreteDecisionXLSTMModel(nn.Module):
    """Policy `forward` on the inference-cache path, batched over B envs.

    forward(states[B,T,204], actions[B,T,A], rewards[B,T,1], returns_to_go[B,T,1], timesteps[B,T], attention_mask,
            ..., past_key_values, use_inference_cache=True) -> output with .action_preds [B,1,A], .action_logits,
            .past_key_values, .last_hidden_state — only the LAST timestep is consumed, exactly as
            `compute_inputs` does when the cache is warm (online_decision_transformer_model.py:466-470); on the cold
            first call the reference embeds all T but `handle_inference_cache` trims to the last 3 tokens
            (decision_xlstm.py:225-229), i.e. to the last timestep as well (pinned by tests/golden/ref_policy_forward/).
    forward(..., use_inference_cache=False) is the reference's ordinary forward: outputs for all T timesteps from a zero
            state, computed in one chunkwise pass (`_forward_sequence`).

    `state_dict` may be given at construction (then it is loaded straight away) or later through `load_state_dict`,
    the order the reference's agent uses; hot-path keys missing at the first call raise KeyError.
    """

    def __init__(self, config, state_dict: Optional[Dict[str, torch.Tensor]] = None, max_batch: int = 1,
                 device=None, mode: int = L.XL_MODE_FUSED, use_graph: bool = True, image_shape=(3, 64, 64),
                 img_is_encoded: bool = False, with_image: Optional[bool] = None):
        super().__init__()
        cfg = config_from_reference(config)
        self.config = cfg
        self.cfg = cfg
        self.max_batch = int(max_batch)
        self._device = torch.device(device) if device is not None else None
        self._engine: Optional[XLSTMEngine] = None
        self._loaded = set()
        self.mode = mode
        self.use_graph = use_graph
        self.image_shape = tuple(image_shape) if image_shape is not None else None
        self.img_is_encoded = img_is_encoded
        self.image_max_frames = 2048        # frames per ImpalaCNN call on the sequence forward (embed_frames)
        d = cfg.d
        # LRAM-side modules, reference names (online_decision_transformer_model.py:92-94, multi_domain...:47-49,67-81)
        self.embed_state = nn.Linear(cfg.state_dim, d)
        self.embed_return = nn.Linear(1, d)
        self.embed_rewards = nn.Linear(1, d)
        self.embed_ln = nn.LayerNorm(d, eps=cfg.embed_ln_eps)
        self.action_net = nn.Sequential(nn.Linear(d, cfg.head_out))
        self.encoder = FusedXLSTMEncoder(config=cfg, mode=mode, max_batch=max_batch, device=device)
        self.encoder._engine_provider = lambda: self.engine     # one handle, one device copy of the block weights
        sd = strip_checkpoint_prefixes(state_dict) if state_dict is not None else None
        if with_image is None:
            with_image = sd is not None and any(k.startswith("embed_image.") for k in sd)
        # embed_image (ImpalaCNN, multi_domain_discrete_dt_model.py:38-46) stays a PyTorch/cuDNN module
        # (SURVEY.md §8 a12) feeding the CUDA path with state embeddings
        self.embed_image = ImpalaCNN(self.image_shape, d).eval() if with_image else None
        for p in self.parameters():
            p.requires_grad_(False)
        self.is_discrete = True            # policy built on a Discrete-action train env (SURVEY App. C.5)
        self.tok_to_pos = {"s": 0, "rtg": 1, "r": 2}
        self.tok_to_pred_pos = {"s": 2, "rtg": 0, "a": 1, "r": 1}
        self.tok_a_target_only, self.shared_a_head = False, True
        self.action_tokenizer = make_tokenizer("minmax", {"vocab_size": cfg.action_channels,
                                                          "shift": cfg.discrete_actions})
        self._stage: Dict[tuple, dict] = {}
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._after_load())
        if sd is not None:
            self.load_state_dict(sd)
            _ = self.engine                                     # weights given up front: build (and fail) now

    @classmethod
    def from_reference_args(cls, config, observation_space=None, action_space=None, stochastic_policy=False,
                            action_channels=256, discrete_actions=18, state_dim=204, image_shape=(3, 64, 64),
                            max_act_dim=None, img_is_encoded=False, max_batch: int = 1, **model_kwargs):
        """Constructor with the reference's signature `Model(config, observation_space, action_space, **model_kwargs)`
        (src/algos/builder.py:95-99) for `MODEL_CLASSES["MDDXLSTM"]` (src/algos/__init__.py:49-53). Options that
        change the token layout away from the multi_domain configuration raise."""
        want = dict(reward_condition=True, tokenize_a=True, tokenize_rtg=False, relative_pos_embds=False,
                    use_time_embds=False, action_condition=False, shared_a_head=True)
        for k, v in want.items():
            if k in model_kwargs and bool(model_kwargs[k]) != v:
                raise NotImplementedError(f"{k}={model_kwargs[k]!r}: only the multi_domain layout (s, rtg, r) with a "
                                          "shared action head is implemented (model_kwargs/multi_domain.yaml)")
        if stochastic_policy:
            raise NotImplementedError("stochastic policy is not implemented for the multi-domain discrete model "
                                      "(multi_domain_discrete_dt_model.py:73-74 raises as well)")
        kw = dict(action_channels=action_channels, discrete_actions=discrete_actions, state_dim=state_dim)
        if max_act_dim is not None:
            kw["act_dim"] = int(max_act_dim)
        cfg = config_from_reference(config, **kw)
        return cls(cfg, None, max_batch=max_batch, image_shape=image_shape, img_is_encoded=img_is_encoded,
                   with_image=image_shape is not None)

    # ---- weights / engine -------------------------------------------------------------------------------------------
    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        """Accepts a full reference checkpoint: DDP / torch.compile prefixes are stripped
        (decision_transformer_sb3.py:1138,1153-1158), tensors the path never reads are ignored, `embed_image.*` is
        taken when this policy has the image front-end. Missing hot-path keys raise KeyError (strict) ."""
        sd = strip_checkpoint_prefixes(state_dict)
        sd = {k: v for k, v in sd.items() if not k.startswith(_OFF_PATH_PREFIXES)}
        if self.embed_image is None:
            sd = {k: v for k, v in sd.items() if not k.startswith("embed_image.")}
        own = set(self.state_dict().keys())
        missing = sorted(own - set(sd))
        unexpected = sorted(set(sd) - own)
        if strict and missing:
            raise KeyError(f"state_dict is missing {missing[0]}" + (f" (+{len(missing) - 1} more)" if len(missing) > 1 else ""))
        if strict and unexpected:
            raise KeyError(f"unexpected key {unexpected[0]} in state_dict" +
                           (f" (+{len(unexpected) - 1} more)" if len(unexpected) > 1 else ""))
        self._loaded |= set(sd) & own
        return super().load_state_dict({k: v for k, v in sd.items() if k in own}, strict=False, assign=assign)

    def _after_load(self):
        self.invalidate_engine()

    def invalidate_engine(self):
        if self._engine is not None:
            self._engine.close()
            self._engine = None
        self._stage.clear()

    @property
    def engine(self) -> XLSTMEngine:
        if self._engine is None:
            sd = {k: v for k, v in self.state_dict().items() if not k.startswith("embed_image.")}
            p = self.embed_state.weight
            dev = self._device or (p.device if p.is_cuda else None)
            self._engine = XLSTMEngine(self.cfg, sd, max_batch=self.max_batch, device=dev)
            if self.embed_image is not None:
                self.embed_image.to(self._engine.device)
        return self._engine

    def engine_for(self, B: int) -> XLSTMEngine:
        """The engine, rebuilt with room for B envs when it has less."""
        if B > self.engine.max_batch:
            self.max_batch = self.encoder.max_batch = B
            self.invalidate_engine()
        return self.engine

    @property
    def device(self):
        return self.engine.device

    def _staging(self, B: int, discrete: bool, state_embeds: bool) -> dict:
        """Persistent per-(B, head, input kind) input and output buffers: a CUDA graph is keyed on its pointers, so graph
        replay needs the SAME tensors on every call (fresh allocations would re-capture a graph per call)."""
        key = (B, discrete, state_embeds)
        st = self._stage.get(key)
        if st is None:
            cfg, dev = self.cfg, self.engine.device
            f32 = dict(dtype=torch.float32, device=dev)
            st = {"states": torch.zeros(B, cfg.d if state_embeds else cfg.state_dim, **f32),
                  "rtg": torch.zeros(B, **f32), "rewards": torch.zeros(B, **f32),
                  "out": {"action_tokens": torch.zeros(B, cfg.act_dim, dtype=torch.int32, device=dev),
                          "action_preds": torch.zeros(B, cfg.act_dim, **f32),
                          "action_logits": torch.empty(B, cfg.num_actions if discrete else cfg.head_out, **f32),
                          "last_hidden_state": torch.empty(B, cfg.tokens_per_step, cfg.d, **f32)}}
            self._stage[key] = st
        return st

    # ---- forward (online_decision_transformer_model.py:326-390) ---------------------------------------------------
    @torch.no_grad()
    def forward(self, states=None, actions=None, rewards=None, returns_to_go=None, timesteps=None,
                attention_mask=None, output_hidden_states=None, output_attentions=None, return_dict=None,
                deterministic=True, with_log_probs=False, prompt=None, task_id=None, ddp_kwargs=None,
                context_trjs=None, inference_params=None, past_key_values=None, use_inference_cache=False):
        if prompt is not None or context_trjs is not None:
            raise NotImplementedError("prompts / retrieval contexts are out of scope")
        if not use_inference_cache:
            return self._forward_sequence(states, actions, rewards, returns_to_go)
        cfg = self.cfg
        B = states.shape[0]
        engine = self.engine_for(B)
        dev = engine.device
        state_embeds = False
        if states.dim() == 5:
            # image observations [B, T, C, H, W], raw 0..255 whatever the dtype: /255 (unconditionally, as embed_inputs
            # does) + embed_image on the newest frame (online_decision_transformer_model.py:522-526,
            # discrete_decision_transformer_model.py:187-203)
            if self.embed_image is None:
                raise ValueError("image observations need embed_image.* weights in the state_dict")
            s_last = self.embed_image(scale_frames(states[:, -1].to(dev)))
            state_embeds = True
        elif states.dim() == 3 and self.img_is_encoded and states.shape[-1] == cfg.d:
            s_last = states[:, -1]
            state_embeds = True                     # discrete_decision_transformer_model.py:185-186
        elif states.dim() != 3:
            raise ValueError(f"states must be [B,T,{cfg.state_dim}] or [B,T,C,H,W], got {tuple(states.shape)}")
        elif states.shape[-1] != cfg.state_dim:
            raise ValueError(f"states must be padded to {cfg.state_dim} (DecisionXLSTM.pad_inputs)")
        else:
            s_last = states[:, -1]
        # is_discrete passed to the head = not actions.is_floating_point(); actions become int64 only for 1-D
        # action envs (online_decision_transformer_model.py:350-352,364)
        discrete = bool(self.is_discrete and actions is not None and actions.shape[-1] == 1)
        if past_key_values is None:
            cache = engine.new_state(B)
        elif isinstance(past_key_values, StateCache):
            cache = past_key_values
            cache.engine = engine
        else:
            cache = engine.new_state(B)
            cache.load_past_key_values(past_key_values)
        if cache.B != B:
            raise ValueError(f"past_key_values holds {cache.B} envs, inputs have batch {B}")
        st = self._staging(B, discrete, state_embeds)
        st["states"].copy_(s_last.reshape(B, -1), non_blocking=True)
        st["rtg"].copy_(returns_to_go[:, -1].reshape(B), non_blocking=True)
        if rewards is not None:
            st["rewards"].copy_(rewards[:, -1].reshape(B), non_blocking=True)
        else:
            st["rewards"].zero_()
        flags = (L.XL_FLAG_DISCRETE if discrete else 0) | (L.XL_FLAG_GRAPH if self.use_graph else 0)
        out = engine.policy_step(cache, st["states"], st["rtg"], st["rewards"], mode=self.mode, flags=flags,
                                 out=st["out"], state_embeds=state_embeds)
        tokens = out["action_tokens"].to(torch.long)
        if discrete:
            action_preds = tokens[:, :1].reshape(B, 1, 1)
            logits = out["action_logits"].clone().view(B, 1, 1, cfg.num_actions)
        else:
            action_preds = out["action_preds"].clone().view(B, 1, cfg.act_dim)
            logits = out["action_logits"].clone().view(B, 1, cfg.act_dim, cfg.num_actions)
        return _Output(last_hidden_state=out["last_hidden_state"].clone(), action_preds=action_preds,
                       action_logits=logits, action_tokens=tokens, past_key_values=cache,
                       state_preds=None, return_preds=None, reward_preds=None, action_log_probs=None,
                       hidden_states=None, attentions=None, entropy=None, prompt_infos=None, cross_attentions=None)

    def _forward_sequence(self, states, actions, rewards, returns_to_go):
        """`forward(use_inference_cache=False)`: the reference's ordinary forward over all T timesteps, each read at its
        rtg token (SURVEY.md a10/a11), from a fresh zero state; no cache is kept (`past_key_values=None`). Runs as one
        `XLSTMEngine.policy_forward`. Returns action_preds [B,T,A] (discrete [B,T,1]), action_logits [B,T,A,num_actions]
        (discrete [B,T,1,num_actions]) and action_tokens. `last_hidden_state` is None: the sequence forward returns no
        hidden states. `attention_mask` is not read, as the reference's encoder does not read it. Rewards None = 0.
        Image observations take the cache path's two forms: raw frames [B,T,C,H,W] (0..255) through embed_image
        (`image_encoder.embed_frames`, in slices of `image_max_frames` frames), or [B,T,d] embeddings with
        `img_is_encoded`; both run as one `policy_forward(state_embeds=True)`."""
        cfg = self.cfg
        encoded = states.dim() == 3 and self.img_is_encoded and states.shape[-1] == cfg.d
        if states.dim() == 5 and self.embed_image is None:
            raise NotImplementedError("image observations on the sequence forward need embed_image.* weights")
        if states.dim() == 3 and not encoded and states.shape[-1] != cfg.state_dim:
            raise ValueError(f"states must be padded to {cfg.state_dim} (DecisionXLSTM.pad_inputs)")
        if states.dim() not in (3, 5):
            raise ValueError(f"states must be [B,T,{cfg.state_dim}] or [B,T,C,H,W], got {tuple(states.shape)}")
        B, T = states.shape[:2]
        engine = self.engine_for(B)
        dev = engine.device
        discrete = bool(self.is_discrete and actions is not None and actions.shape[-1] == 1)
        if states.dim() == 5:
            st = embed_frames(self.embed_image, states, max_frames=self.image_max_frames)
        else:
            st = states.to(dev, torch.float32).contiguous()
        rtg = returns_to_go.to(dev, torch.float32).reshape(B, T).contiguous()
        rew = None if rewards is None else rewards.to(dev, torch.float32).reshape(B, T).contiguous()
        out = engine.policy_forward(engine.new_state(B), st, rtg, rew, discrete=discrete, want_logits=True,
                                    state_embeds=states.dim() == 5 or encoded)
        tokens = out["action_tokens"].to(torch.long)
        if discrete:
            action_preds = tokens[:, :, :1]
            logits = out["action_logits"].view(B, T, 1, cfg.num_actions)
        else:
            action_preds = out["action_preds"]
            logits = out["action_logits"].view(B, T, cfg.act_dim, cfg.num_actions)
        return _Output(last_hidden_state=None, action_preds=action_preds, action_logits=logits, action_tokens=tokens,
                       past_key_values=None, state_preds=None, return_preds=None, reward_preds=None,
                       action_log_probs=None, hidden_states=None, attentions=None, entropy=None, prompt_infos=None,
                       cross_attentions=None)


def sample_from_logits(logits: torch.Tensor, temperature: float = 1.0, top_k: int = 0, top_p: float = 0.5):
    """Action sampling of `a_sample_kwargs` (src/algos/models/model_utils.py:7-32): quantile cut at `top_p`, optional
    top-k, categorical sample at `temperature * logits` (the reference multiplies), in fp64. Returns token ids."""
    logits = logits.double()
    if top_p > 0.0:
        percentile = torch.quantile(logits, top_p, dim=-1)
        if (percentile != logits.max()).all() if percentile.dim() else percentile != logits.max():
            logits = torch.where(logits > percentile.unsqueeze(-1), logits, -float("inf"))
    top_indices = None
    if top_k > 0:
        logits, top_indices = torch.topk(logits, top_k)
    sample = torch.distributions.Categorical(logits=temperature * logits).sample()
    if top_indices is not None:
        shape = sample.shape
        flat = sample.flatten()
        sample = top_indices.reshape(-1, top_k)[torch.arange(len(flat), device=flat.device), flat].reshape(shape)
    return sample


@dataclasses.dataclass
class _ReplayBufferDims:
    max_state_dim: Optional[int] = 204
    max_act_dim: Optional[int] = 8
    seqs_per_sample: int = 1


class DiscreteDecisionXLSTM:
    """Agent-side `predict` for ONE env (B == 1), as the reference's rollout loop calls it
    (src/callbacks/evaluation.py:134-139), plus `predict_batch`, the same computation for B envs at once (used by
    `lram_b200.rollout.custom_evaluate_policy`). Carries what the loop reads from the agent: `past_key_values`,
    `use_inference_cache`, `eval_context_len`, `persist_context`, `compute_target_return_val`,
    `get_reward_scale_for_env`.

    `a_sample_kwargs` samples the actions as the reference does (`sample_from_logits` on the step's logits, torch's
    global RNG). Setting `a_sample_seed` as well moves the draw onto the device: the policy's engine is armed with
    those kwargs (`XLSTMEngine.set_sampling`, a Philox stream keyed on the seed) and `predict` / `predict_batch` return
    the step's sampled action tokens, with the shape and dtype of the torch path. The two paths differ in one place:
    the torch path's top-p guard (`percentile != max`, all rows) spans the whole batch of `predict_batch`, the device
    path takes it per env, as the reference's one call per env does."""

    def __init__(self, policy: MultiDomainDiscreteDecisionXLSTMModel, use_inference_cache: bool = True,
                 state_mean=None, state_std=None, reset_inf_cache_freq: Optional[int] = None,
                 target_return: float = 1.0, reward_scale: float = 1.0, persist_context: bool = False,
                 eval_context_len: int = 5, a_sample_kwargs: Optional[dict] = None,
                 a_sample_seed: Optional[int] = None):
        self.policy = policy
        self.device = policy.device
        self.use_inference_cache = use_inference_cache
        self.past_key_values: Optional[Any] = None
        self.replay_buffer = _ReplayBufferDims(policy.config.state_dim, policy.config.act_dim)
        self.state_mean, self.state_std = state_mean, state_std
        self.reset_inf_cache_freq = reset_inf_cache_freq
        self.target_return_type = "fixed"
        self.target_return = target_return          # already divided by reward_scale (src/algos/builder.py:86-88)
        self._reward_scale = reward_scale
        self.persist_context = persist_context
        self.eval_context_len = eval_context_len
        self.a_sample_kwargs = a_sample_kwargs
        self.a_sample_seed = a_sample_seed
        self._sampler_engine = None                 # weakref to the engine armed with the device sampler
        self.s_proj_raw = False
        self.ddp_kwargs: Dict[str, Any] = {}

    # decision_transformer_sb3.py:373-382, 542-567 (the "fixed" target-return type; the tables of per-env targets
    # behind "predefined" are env metadata, out of scope)
    def get_reward_scale_for_env(self, envid=None):
        if isinstance(self._reward_scale, dict) and envid is not None:
            return self._reward_scale[envid]
        return self._reward_scale

    def compute_target_return_val(self, env=None, task_id=0):
        return self.target_return

    def pad_inputs(self, states, actions, returns_to_go, timesteps, context_len=5, rewards=None):
        """decision_xlstm.py:11-28 (cache mode): no time padding; zero-pad state -> 204 and action -> 8."""
        if not self.use_inference_cache:
            raise NotImplementedError("only the inference-cache path is implemented")
        attention_mask = torch.ones(actions.shape[1], device=self.device, dtype=torch.long).reshape(1, -1)
        rb = self.replay_buffer
        if rb.max_state_dim is not None and states.dim() == 3 and not self.s_proj_raw:
            pad = rb.max_state_dim - states.shape[-1]
            states = torch.cat([states, torch.zeros((*states.shape[:-1], pad), device=states.device)], dim=-1)
        if rb.max_act_dim is not None and actions.is_floating_point() and states.dim() != 5:
            pad = rb.max_act_dim - actions.shape[-1]
            actions = torch.cat([actions, torch.zeros((*actions.shape[:-1], pad), device=actions.device)], dim=-1)
        return states.float(), actions, returns_to_go.float(), timesteps, attention_mask, rewards

    def predict(self, policy, observation, actions, rewards, returns_to_go, timesteps, state=None,
                episode_start=None, deterministic=True, context_len=5, prompt=None, task_id=None, is_eval=False,
                env_act_dim=None):
        """decision_transformer_sb3.py:621-667."""
        obs_shape, act_dim = observation.shape[1:], actions.shape[-1]
        states = observation.reshape(1, -1, *obs_shape)[:, -context_len:]
        actions = actions.reshape(1, -1, act_dim)[:, -context_len:]
        returns_to_go = returns_to_go.reshape(1, -1, 1)[:, -context_len:]
        timesteps = timesteps.reshape(1, -1)[:, -context_len:]
        if rewards is not None:
            rewards = rewards.reshape(1, -1, 1)[:, -context_len:]
        states, actions, returns_to_go, timesteps, attention_mask, rewards = self.pad_inputs(
            states, actions, returns_to_go, timesteps, context_len=context_len, rewards=rewards)
        if self.state_mean is not None and self.state_std is not None:
            states = (states - self.state_mean) / self.state_std
        a1, a2 = self.get_action_pred(policy, states, actions, rewards, returns_to_go, timesteps, attention_mask,
                                      deterministic, prompt, task_id=task_id, is_eval=is_eval,
                                      env_act_dim=env_act_dim)
        if self.reset_inf_cache_freq is not None:
            cur = int(timesteps[0, -1])
            if cur > 0 and cur % self.reset_inf_cache_freq == 0:
                self.past_key_values = None
        return a1, a2

    def get_action_pred(self, policy, states, actions, rewards, returns_to_go, timesteps, attention_mask,
                        deterministic, prompt, is_eval=False, task_id=None, env_act_dim=None):
        """discrete_decision_transformer_sb3.py:13-72, shared-action-head branch (:60-68)."""
        device_sampling = self._arm_device_sampler(policy, states.shape[0])
        out = policy(states=states, actions=actions, rewards=rewards, returns_to_go=returns_to_go,
                     timesteps=timesteps, attention_mask=attention_mask, return_dict=True,
                     deterministic=deterministic, prompt=prompt, task_id=task_id, ddp_kwargs=self.ddp_kwargs,
                     use_inference_cache=self.use_inference_cache, past_key_values=self.past_key_values)
        if device_sampling:
            action = out.action_tokens[0, :out.action_logits.shape[-2]]
        elif self.a_sample_kwargs is not None:
            action = sample_from_logits(out.action_logits[0, -1], **self.a_sample_kwargs)   # :62-63
        else:
            action = out.action_preds[0, -1]
        if self.use_inference_cache:
            self.past_key_values = out.past_key_values
        if env_act_dim is not None:
            action = action[:env_act_dim]
        return action, action

    def _arm_device_sampler(self, policy, B: int) -> bool:
        """True when actions are drawn on the device; arms the engine that will run a batch of B envs once."""
        if self.a_sample_kwargs is None or self.a_sample_seed is None:
            return False
        engine = policy.engine_for(B)
        if self._sampler_engine is None or self._sampler_engine() is not engine:
            engine.set_sampling(**self.a_sample_kwargs, seed=self.a_sample_seed)
            self._sampler_engine = weakref.ref(engine)
        return True

    @torch.no_grad()
    def predict_batch(self, policy, observations: torch.Tensor, returns_to_go: torch.Tensor, action_dim: int,
                      env_act_dim=None):
        """`predict` for B envs, newest timestep only (what the cache-mode path consumes): observations [B, *obs_shape],
        returns_to_go [B] -> actions [B, env_act_dim]. The recurrent state of all B envs is `self.past_key_values`."""
        B = observations.shape[0]
        states = observations.reshape(B, 1, *observations.shape[1:]).to(self.device)
        actions = torch.zeros(B, 1, action_dim, device=self.device)          # evaluation.py:131 placeholder
        rewards = torch.zeros(B, 1, 1, device=self.device)                   # evaluation.py:132 placeholder
        rtg = returns_to_go.reshape(B, 1, 1).to(self.device)
        timesteps = torch.zeros(B, 1, dtype=torch.long, device=self.device)
        states, actions, rtg, timesteps, _, rewards = self.pad_inputs(states, actions, rtg, timesteps, rewards=rewards)
        if self.state_mean is not None and self.state_std is not None:
            states = (states - self.state_mean) / self.state_std
        device_sampling = self._arm_device_sampler(policy, B)
        out = policy(states=states, actions=actions, rewards=rewards, returns_to_go=rtg, timesteps=timesteps,
                     attention_mask=torch.ones(B, 1, dtype=torch.long, device=self.device), return_dict=True,
                     deterministic=True, prompt=None, task_id=None, ddp_kwargs=self.ddp_kwargs,
                     use_inference_cache=True, past_key_values=self.past_key_values)
        self.past_key_values = out.past_key_values
        if device_sampling:
            act = out.action_tokens[:, :out.action_logits.shape[-2]]
        elif self.a_sample_kwargs is not None:
            act = sample_from_logits(out.action_logits[:, -1], **self.a_sample_kwargs)
        else:
            act = out.action_preds[:, -1]
        return act[:, :env_act_dim] if env_act_dim is not None else act
