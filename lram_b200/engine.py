"""Host side of the CUDA path: one `XLSTMEngine` per GPU/process.

Owns (as PyTorch tensors — PyTorch is only the allocator / stream provider here):
  * the packed weights on the device (bf16 GEMM matrices, fp32 everything else),
  * the per-GPU recurrent state cache (C, n, m, conv of every block for B envs, one buffer),
and calls the C-ABI library (include/xlstm_b200.h) through ctypes with raw pointers + the current stream.

Reference counterparts: `xLSTMEncoder` (src/algos/models/decision_xlstm.py:119-172) for the encoder step,
`MultiDomainDiscreteDecisionXLSTMModel.forward` for the policy step, and the `past_key_values` dict
({"block_i": {"mlstm_state": (C, n, m), "conv_state": (conv,)}}) for import/export of the state.
"""
from __future__ import annotations

import ctypes as C
import functools
import math
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib as L
from .config import XLSTMPolicyConfig
from .synth import is_bf16_weight

_BLOCK_KEYS = {
    "xlstm_norm.weight": "XLSTM_NORM",
    "xlstm.proj_up.weight": "PROJ_UP",
    "xlstm.q_proj.weight": "Q_PROJ",
    "xlstm.k_proj.weight": "K_PROJ",
    "xlstm.v_proj.weight": "V_PROJ",
    "xlstm.conv1d.conv.weight": "CONV_W",
    "xlstm.conv1d.conv.bias": "CONV_B",
    "xlstm.mlstm_cell.igate.weight": "IGATE_W",
    "xlstm.mlstm_cell.igate.bias": "IGATE_B",
    "xlstm.mlstm_cell.fgate.weight": "FGATE_W",
    "xlstm.mlstm_cell.fgate.bias": "FGATE_B",
    "xlstm.mlstm_cell.outnorm.weight": "OUTNORM",
    "xlstm.learnable_skip": "SKIP",
    "xlstm.proj_down.weight": "PROJ_DOWN",
}
# sLSTM block of an xLSTM[a:b] stack (xlstm v1.0.x sLSTMLayer + GatedFeedForward state_dict names). NB the module
# named `fgate` feeds the INPUT gate and `igate` the FORGET gate (quirk of sLSTMLayer.forward, see the oracle).
_SLSTM_BLOCK_KEYS = {
    "xlstm_norm.weight": "XLSTM_NORM",
    "xlstm.conv1d.conv.weight": "CONV_W",
    "xlstm.conv1d.conv.bias": "CONV_B",
    "xlstm.fgate.weight": "S_GATE_I",
    "xlstm.igate.weight": "S_GATE_F",
    "xlstm.zgate.weight": "S_GATE_Z",
    "xlstm.ogate.weight": "S_GATE_O",
    "xlstm.slstm_cell._recurrent_kernel_": "S_RECURRENT",
    "xlstm.slstm_cell._bias_": "S_BIAS",
    "xlstm.group_norm.weight": "S_GROUP_NORM",
    "ffn_norm.weight": "FFN_NORM",
    "ffn.proj_up.weight": "FFN_UP",
    "ffn.proj_down.weight": "FFN_DOWN",
}
_POLICY_KEYS = {
    "encoder.layers.post_blocks_norm.weight": "POST_NORM",
    "embed_state.weight": "EMBED_STATE_W",
    "embed_state.bias": "EMBED_STATE_B",
    "embed_return.weight": "EMBED_RETURN_W",
    "embed_return.bias": "EMBED_RETURN_B",
    "embed_rewards.weight": "EMBED_REWARD_W",
    "embed_rewards.bias": "EMBED_REWARD_B",
    "embed_ln.weight": "EMBED_LN_W",
    "embed_ln.bias": "EMBED_LN_B",
    "action_net.0.weight": "HEAD_W",
    "action_net.0.bias": "HEAD_B",
}


def strip_checkpoint_prefixes(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """`load_model_weights` strips DDP / torch.compile prefixes (decision_transformer_sb3.py:1138,1153-1158)."""
    out = {}
    for k, v in sd.items():
        for pref in ("module.", "_orig_mod."):
            while k.startswith(pref):
                k = k[len(pref):]
        k = k.replace("._orig_mod.", ".").replace(".module.", ".")
        out[k] = v
    return out


def slab_width(DH: int) -> int:
    """Column-slab width of the C layout in HBM (include/xlstm_b200.h, xl_state_layout)."""
    return 128 if DH % 128 == 0 else DH


def c_to_slab(c: torch.Tensor) -> torch.Tensor:
    """reference layout C[B,NH,DH(dk),DH(dv)] -> slab-major [B,NH,DH/W,DH,W] (contiguous copy)."""
    B, NH, DH, _ = c.shape
    W = slab_width(DH)
    return c.reshape(B, NH, DH, DH // W, W).permute(0, 1, 3, 2, 4).contiguous()


def c_from_slab(p: torch.Tensor) -> torch.Tensor:
    """slab-major [B,NH,CS,DH,W] -> reference layout [B,NH,DH,DH] (copy)."""
    B, NH, CS, DH, W = p.shape
    return p.permute(0, 1, 3, 2, 4).reshape(B, NH, DH, CS * W)


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(0 if t is None else t.data_ptr())


class StateCache:
    """The recurrent state of B envs on one GPU. Opaque `past_key_values` of the CUDA path."""

    def __init__(self, engine: "XLSTMEngine", B: int):
        self.engine = engine
        self.B = B
        nbytes = engine.lib.xl_state_bytes(engine.handle, B)
        self.buf = torch.zeros(nbytes // 4, dtype=torch.float32, device=engine.device)

    def view(self, layer: int, part: int) -> torch.Tensor:
        off, size = C.c_size_t(), C.c_size_t()
        L.check(self.engine.lib.xl_state_layout(self.engine.handle, self.B, layer, part, C.byref(off), C.byref(size)))
        flat = self.buf[off.value // 4: (off.value + size.value) // 4]
        cfg = self.engine.cfg
        NH, DH = cfg.num_heads, cfg.head_dim
        W = slab_width(DH)
        if cfg.is_slstm(layer):
            shape = {L.XL_STATE_SLSTM: (4, self.B, cfg.d),
                     L.XL_STATE_CONV: (self.B, cfg.conv1d_kernel_size, cfg.d)}[part]
        else:
            shape = {L.XL_STATE_C: (self.B, NH, DH // W, DH, W), L.XL_STATE_N: (self.B, NH, DH),
                     L.XL_STATE_M: (self.B, NH), L.XL_STATE_CONV: (self.B, cfg.conv1d_kernel_size, cfg.inner)}[part]
        return flat.view(*shape)

    def c_logical(self, layer: int) -> torch.Tensor:
        """C of one block in the reference's [B, NH, DH(dk), DH(dv)] layout (a copy; the cache itself is slab-major)."""
        return c_from_slab(self.view(layer, L.XL_STATE_C))

    def nbytes(self) -> int:
        return self.buf.numel() * 4

    # ---- reference-format import / export ------------------------------------------------------
    def to_past_key_values(self) -> Dict[str, Dict[str, tuple]]:
        out = {}
        for i in range(self.engine.cfg.num_blocks):
            if self.engine.cfg.is_slstm(i):
                out[f"block_{i}"] = {"slstm_state": self.view(i, L.XL_STATE_SLSTM).clone(),
                                     "conv_state": (self.view(i, L.XL_STATE_CONV).clone(),)}
                continue
            c = self.c_logical(i)
            n = self.view(i, L.XL_STATE_N).clone().unsqueeze(-1)
            m = self.view(i, L.XL_STATE_M).clone().view(self.B, -1, 1, 1)
            conv = self.view(i, L.XL_STATE_CONV).clone()
            out[f"block_{i}"] = {"mlstm_state": (c, n, m), "conv_state": (conv,)}
        return out

    def load_past_key_values(self, pkv: Dict[str, Dict[str, tuple]]) -> None:
        for i in range(self.engine.cfg.num_blocks):
            st = pkv[f"block_{i}"]
            if self.engine.cfg.is_slstm(i):
                self.view(i, L.XL_STATE_SLSTM).copy_(st["slstm_state"].to(self.buf.device, torch.float32))
                self.view(i, L.XL_STATE_CONV).copy_(st["conv_state"][0].to(self.buf.device, torch.float32))
                continue
            c, n, m = st["mlstm_state"]
            self.view(i, L.XL_STATE_C).copy_(c_to_slab(c.to(self.buf.device, torch.float32)))
            self.view(i, L.XL_STATE_N).copy_(n.to(self.buf.device, torch.float32).reshape(self.B, -1, n.shape[2]))
            self.view(i, L.XL_STATE_M).copy_(m.to(self.buf.device, torch.float32).reshape(self.B, -1))
            self.view(i, L.XL_STATE_CONV).copy_(st["conv_state"][0].to(self.buf.device, torch.float32))


def sampling_params(cfg: XLSTMPolicyConfig, temperature: float = 1.0, top_k: int = 0, top_p: float = 0.5,
                    seed: int = 0, env_id_base: int = 0, env_id_stride: int = 1) -> L.XLSampling:
    """Checked `xl_sampling` for the device sampler; raises ValueError on what the library would reject."""
    temperature, top_p = float(temperature), float(top_p)
    if not (math.isfinite(temperature) and temperature > 0.0):
        raise ValueError(f"temperature={temperature} must be finite and > 0")
    if not 0.0 <= top_p <= 1.0:
        raise ValueError(f"top_p={top_p} outside [0, 1]")
    if not 0 <= int(top_k) <= cfg.num_actions:
        raise ValueError(f"top_k={top_k} outside [0, num_actions={cfg.num_actions}]")
    if int(env_id_base) < 0 or int(env_id_stride) < 1:
        raise ValueError(f"env_id_base={env_id_base} must be >= 0 and env_id_stride={env_id_stride} >= 1")
    if not 0 <= int(seed) < 2 ** 64:
        raise ValueError(f"seed={seed} outside [0, 2^64)")
    return L.XLSampling(temperature=temperature, top_p=top_p, top_k=int(top_k), env_id_base=int(env_id_base),
                        env_id_stride=int(env_id_stride), seed=int(seed))


def check_lengths(lengths, B: int, S: int, what: str = "S") -> np.ndarray:
    """Per-env context lengths of a ragged prefill as the library takes them (a host int32 [B] array): a sequence, an
    ndarray or a CPU integer tensor of B values in [0, S]. Raises ValueError otherwise."""
    if isinstance(lengths, torch.Tensor):
        if lengths.device.type != "cpu":
            raise ValueError(f"lengths must be on the host, got a tensor on {lengths.device}")
        if lengths.dtype.is_floating_point or lengths.dtype.is_complex or lengths.dtype == torch.bool:
            raise ValueError(f"lengths must be integers, got {lengths.dtype}")
        lengths = lengths.numpy()
    arr = np.asarray(lengths)
    if arr.ndim != 1 or arr.shape[0] != B:
        raise ValueError(f"lengths must hold one value per env ({B}), got shape {arr.shape}")
    if arr.dtype == np.bool_ or not np.issubdtype(arr.dtype, np.integer):
        raise ValueError(f"lengths must be integers, got dtype {arr.dtype}")
    if (arr < 0).any() or (arr > S).any():
        raise ValueError(f"lengths must lie in [0, {what}={S}], got min {arr.min()} max {arr.max()}")
    return np.ascontiguousarray(arr, dtype=np.int32)


def _on_device(fn):
    """Run an engine method with the engine's GPU as the current CUDA device: the handle, its workspace, its streams
    and the per-device kernel attributes all belong to `self.device`, whatever device the caller has current."""
    @functools.wraps(fn)
    def wrapped(self, *args, **kwargs):
        if torch.cuda.current_device() == self.device.index:
            return fn(self, *args, **kwargs)
        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)
    return wrapped


class XLSTMEngine:
    """`encoder_only=True` binds the block stack + post_blocks_norm only: the engine behind a `FusedXLSTMEncoder`
    that replaces just `self.encoder` of a reference policy (decision_xlstm.py:188-189); `policy_step*` then raise
    XL_ERR_NOT_READY, `encoder_step` / `prefill` work."""

    def __init__(self, cfg: XLSTMPolicyConfig, state_dict: Dict[str, torch.Tensor], max_batch: int,
                 device: Optional[torch.device] = None, encoder_only: bool = False):
        if not torch.cuda.is_available():
            raise RuntimeError("XLSTMEngine needs a CUDA device: the xlstm_b200 path has no CPU fallback")
        cfg.validate()
        self.cfg = cfg
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError(f"XLSTMEngine needs a CUDA device, got {self.device}: there is no CPU fallback")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.encoder_only = bool(encoder_only)
        self.max_batch = int(max_batch)
        self.lib = L.load()
        if self.lib.xl_abi_version() != L.XL_ABI_VERSION:
            raise RuntimeError("libxlstm_b200.so ABI mismatch")
        c = L.XLConfig(
            embedding_dim=cfg.d, num_blocks=cfg.num_blocks, num_heads=cfg.num_heads, inner_dim=cfg.inner,
            conv_kernel=cfg.conv1d_kernel_size, qkv_blocksize=cfg.qkv_proj_blocksize, state_dim=cfg.state_dim,
            act_dim=cfg.act_dim, action_channels=cfg.action_channels, discrete_actions=cfg.discrete_actions,
            tokens_per_step=cfg.tokens_per_step, action_token_pos=cfg.action_token_pos, max_batch=self.max_batch,
            ln_eps=cfg.ln_eps, cell_eps=cfg.cell_eps, embed_ln_eps=cfg.embed_ln_eps, tok_min_val=-1.0,
            tok_max_val=1.0, slstm_mask_lo=cfg.slstm_mask & 0xFFFFFFFF, slstm_mask_hi=cfg.slstm_mask >> 32,
            ffn_dim=cfg.ffn_dim if cfg.slstm_at else 0)
        self.handle = C.c_void_p()
        with torch.cuda.device(self.device):
            L.check(self.lib.xl_create(C.byref(c), C.byref(self.handle)))
        self._weights = []          # keep device tensors alive
        with torch.cuda.device(self.device):
            self._bind_all(strip_checkpoint_prefixes(state_dict))
            L.check((self.lib.xl_encoder_weights_ready if self.encoder_only else self.lib.xl_weights_ready)(self.handle))

    # ---- weights ----------------------------------------------------------------------------------
    def _bind(self, layer: int, slot: str, t: torch.Tensor, bf16: bool):
        t = t.detach().to(self.device, torch.bfloat16 if bf16 else torch.float32).contiguous()
        self._weights.append(t)
        L.check(self.lib.xl_bind_weight(self.handle, layer, L.W[slot], _ptr(t), 1 if bf16 else 0, t.numel()))

    def _bind_all(self, sd):
        cfg = self.cfg
        for i in range(cfg.num_blocks):
            slstm = cfg.is_slstm(i)
            for key, slot in (_SLSTM_BLOCK_KEYS if slstm else _BLOCK_KEYS).items():
                name = f"encoder.layers.blocks.{i}.{key}"
                if name not in sd:
                    raise KeyError(f"state_dict is missing {name}")
                t = sd[name]
                if slot == "CONV_W":
                    t = t.reshape(cfg.d if slstm else cfg.inner, cfg.conv1d_kernel_size)
                self._bind(i, slot, t, is_bf16_weight(name))
        kpad = self.lib.xl_state_dim_padded(self.handle)
        for name, slot in _POLICY_KEYS.items():
            if self.encoder_only and slot != "POST_NORM":
                continue
            if name not in sd:
                raise KeyError(f"state_dict is missing {name}")
            t = sd[name]
            if slot == "EMBED_STATE_W":
                w = torch.zeros(cfg.d, kpad, dtype=torch.float32)
                w[:, : cfg.state_dim] = t.detach().float().cpu()
                t = w
            elif slot in ("EMBED_RETURN_W", "EMBED_REWARD_W"):
                t = t.reshape(-1)
            self._bind(-1, slot, t, is_bf16_weight(name))

    # ---- state ------------------------------------------------------------------------------------
    def new_state(self, B: int) -> StateCache:
        if B > self.max_batch:
            raise ValueError(f"B={B} > max_batch={self.max_batch}")
        return StateCache(self, B)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @_on_device
    def reset(self, state: StateCache, mask: Optional[torch.Tensor] = None):
        if mask is not None:
            mask = mask.to(self.device, torch.uint8).contiguous()
            assert mask.numel() == state.B
        L.check(self.lib.xl_state_reset(self.handle, _ptr(state.buf), _ptr(mask), state.B, self._stream()))

    # ---- compute ----------------------------------------------------------------------------------
    @_on_device
    def encoder_step(self, state: StateCache, x: torch.Tensor, mode: int = L.XL_MODE_FUSED, flags: int = 0,
                     out: Optional[torch.Tensor] = None):
        """x [B,T,d] fp32 cuda -> last_hidden_state [B,T,d]; state advanced in place. With XL_FLAG_GRAPH the step is
        replayed from a CUDA graph keyed on (state, x, out): pass the same tensors every step."""
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 3 and x.shape[0] == state.B
        x = x.contiguous()
        if out is None:
            out = torch.empty_like(x)
        assert out.is_contiguous() and out.shape == x.shape and out.dtype == torch.float32
        L.check(self.lib.xl_encoder_step(self.handle, _ptr(state.buf), _ptr(x), _ptr(out), x.shape[0], x.shape[1],
                                         mode, flags, self._stream()))
        return out

    def prefill(self, state: StateCache, x: torch.Tensor, want_hidden: bool = True, flags: int = 0, lengths=None):
        """Context prefill of the encoder: x [B,S,d] fp32 cuda (embedded tokens) -> last_hidden_state [B,S,d]
        (or None); state advanced by S tokens, exactly as S recurrent steps would (xl_prefill).
        `lengths` (B ints in [0, S]: sequence, ndarray or CPU tensor): env b advances by its first lengths[b] tokens
        only, an env with 0 keeps its state, rows from lengths[b] on are never read and come back as 0
        (xl_prefill_ragged). Checked before anything reaches the library."""
        lens = None if lengths is None else check_lengths(lengths, state.B, x.shape[1], "S")
        return self._prefill(state, x, want_hidden, flags, lens)

    @_on_device
    def _prefill(self, state, x, want_hidden, flags, lens):
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 3 and x.shape[0] == state.B
        x = x.contiguous()
        out = torch.empty_like(x) if want_hidden else None
        if lens is None:
            L.check(self.lib.xl_prefill(self.handle, _ptr(state.buf), _ptr(x), _ptr(out), x.shape[0], x.shape[1],
                                        flags, self._stream()))
        else:
            L.check(self.lib.xl_prefill_ragged(self.handle, _ptr(state.buf), _ptr(x), _ptr(out),
                                               lens.ctypes.data_as(C.c_void_p), x.shape[0], x.shape[1], flags,
                                               self._stream()))
        return out

    def _check_state_embeds(self, states, B: int):
        """`states` of a sequence call with state_embeds=True: fp32 [B, Tn, d] on this engine's device."""
        want = f"an fp32 tensor [B={B}, Tn, d={self.cfg.d}] on {self.device}"
        if not isinstance(states, torch.Tensor):
            raise ValueError(f"state embeddings must be {want}, got {type(states).__name__}")
        if states.dim() != 3 or states.shape[0] != B or states.shape[2] != self.cfg.d:
            raise ValueError(f"state embeddings must be {want}, got shape {tuple(states.shape)}")
        if states.dtype != torch.float32:
            raise ValueError(f"state embeddings must be {want}, got {states.dtype}")
        if states.device != self.device:
            raise ValueError(f"state embeddings must be {want}, got a tensor on {states.device}")

    @staticmethod
    def _embeds_operand(states: torch.Tensor) -> torch.Tensor:
        """Contiguous and 16-byte aligned, as the _embeds entries load rows as float4."""
        states = states.contiguous()
        return states.clone() if states.data_ptr() % 16 else states

    def policy_prefill(self, state: StateCache, states: torch.Tensor, rtg: torch.Tensor,
                       rewards: Optional[torch.Tensor] = None, flags: int = 0, lengths=None,
                       state_embeds: bool = False):
        """Warm the recurrent state with Tn timesteps of context per env: states [B,Tn,state_dim], rtg [B,Tn],
        rewards [B,Tn] or None (= the 0 placeholder the rollout feeds). No action outputs (xl_policy_prefill).
        `lengths` (B ints in [0, Tn]): env b takes its first lengths[b] timesteps only, an env with 0 keeps its state
        (xl_policy_prefill_ragged). With `state_embeds=True`, `states` is instead the state-token embedding of every
        timestep, fp32 [B,Tn,d] on this engine's device (image observations: `image_encoder.embed_frames`), and
        embed_state is skipped (xl_policy_prefill_embeds). Checked before anything reaches the library."""
        if state_embeds:
            self._check_state_embeds(states, state.B)
        lens = None if lengths is None else check_lengths(lengths, state.B, states.shape[1], "Tn")
        self._seq_call(state, states, rtg, rewards, lens, flags, state_embeds)

    @_on_device
    def _seq_call(self, state, states, rtg, rewards, lens, flags, state_embeds, outputs=None):
        """The one place a policy sequence call reaches the library: the prefill (outputs None) or the forward
        (outputs: an XLSeqOutputs), from raw states or state embeddings, uniform (lens None) or ragged."""
        B, Tn = state.B, states.shape[1]
        assert states.is_cuda and states.dtype == torch.float32 and tuple(states.shape) == \
            (B, Tn, self.cfg.d if state_embeds else self.cfg.state_dim)
        assert rtg.is_cuda and rtg.dtype == torch.float32 and rtg.numel() == B * Tn
        states = self._embeds_operand(states) if state_embeds else states.contiguous()
        rtg = rtg.contiguous()
        if rewards is not None:
            rewards = rewards.to(self.device, torch.float32).contiguous()
            assert rewards.numel() == B * Tn
        args = (self.handle, _ptr(state.buf), _ptr(states), _ptr(rtg), _ptr(rewards))
        lp = None if lens is None else lens.ctypes.data_as(C.c_void_p)
        if outputs is not None:
            fn = self.lib.xl_policy_forward_embeds if state_embeds else self.lib.xl_policy_forward
            rc = fn(*args, lp, B, Tn, C.byref(outputs), flags, self._stream())
        elif state_embeds:
            rc = self.lib.xl_policy_prefill_embeds(*args, lp, B, Tn, flags, self._stream())
        elif lens is None:
            rc = self.lib.xl_policy_prefill(*args, B, Tn, flags, self._stream())
        else:
            rc = self.lib.xl_policy_prefill_ragged(*args, lp, B, Tn, flags, self._stream())
        L.check(rc)

    def policy_forward(self, state: StateCache, states: torch.Tensor, rtg: torch.Tensor,
                       rewards: Optional[torch.Tensor] = None, lengths=None, discrete: bool = False,
                       targets: Optional[torch.Tensor] = None, want_logits: bool = False,
                       state_embeds: bool = False) -> dict:
        """Action outputs of every timestep of whole trajectories in one chunkwise pass (xl_policy_forward): what
        `policy_step` would return at each timestep when stepped from `state` over states [B,Tn,state_dim], rtg [B,Tn],
        rewards [B,Tn] or None (= 0). The state ends where `policy_prefill` on the same arguments leaves it.
        Returns "action_tokens" (int32) and "action_preds" [B,Tn,act_dim] (argmax, never sampled; discrete: column 0,
        the other columns -1 / 0), with `want_logits` "action_logits" [B,Tn,n_out] (n_out = num_actions when discrete,
        act_dim * num_actions otherwise), and with `targets` (an integer tensor [B,Tn,act_dim] on this engine's device,
        values in [-1, num_actions); -1 = a padded action dim, scored 0) "action_logprobs" [B,Tn,act_dim]: the log-softmax
        of each action row's logits at the target (discrete: column 0). `lengths` (B ints in [0, Tn]) gives env b its
        first lengths[b] timesteps only; outputs past them are -1 / 0 and an env with 0 keeps its state.
        With `state_embeds=True`, `states` is the state-token embedding of every timestep, fp32 [B,Tn,d] on this
        engine's device (image observations: `image_encoder.embed_frames`), as `policy_step(state_embeds=True)` takes
        it (xl_policy_forward_embeds).
        Lengths, targets and embeddings are checked before anything reaches the library; the range check of `targets`
        costs one device reduction and a synchronisation."""
        cfg = self.cfg
        if state_embeds:
            self._check_state_embeds(states, state.B)
        B, Tn = state.B, states.shape[1]
        lens = None if lengths is None else check_lengths(lengths, B, Tn, "Tn")
        if targets is not None:
            if not isinstance(targets, torch.Tensor):
                raise ValueError(f"targets must be a tensor, got {type(targets).__name__}")
            if targets.dtype.is_floating_point or targets.dtype.is_complex or targets.dtype == torch.bool:
                raise ValueError(f"targets must be integers, got {targets.dtype}")
            if tuple(targets.shape) != (B, Tn, cfg.act_dim):
                raise ValueError(f"targets must have shape {(B, Tn, cfg.act_dim)}, got {tuple(targets.shape)}")
            if targets.device != self.device:
                raise ValueError(f"targets must be on {self.device}, got {targets.device}")
            if targets.numel():
                lo, hi = (int(v) for v in torch.aminmax(targets))
                if lo < -1 or hi >= cfg.num_actions:
                    raise ValueError(f"targets must lie in [-1, num_actions={cfg.num_actions}), got min {lo} max {hi}")
        return self._policy_forward(state, states, rtg, rewards, lens, discrete, targets, want_logits, state_embeds)

    @_on_device
    def _policy_forward(self, state, states, rtg, rewards, lens, discrete, targets, want_logits, state_embeds=False):
        cfg = self.cfg
        B, Tn = state.B, states.shape[1]
        out = {"action_tokens": torch.empty(B, Tn, cfg.act_dim, dtype=torch.int32, device=self.device),
               "action_preds": torch.empty(B, Tn, cfg.act_dim, dtype=torch.float32, device=self.device)}
        if want_logits:
            n = cfg.num_actions if discrete else cfg.head_out
            out["action_logits"] = torch.empty(B, Tn, n, dtype=torch.float32, device=self.device)
        if targets is not None:
            targets = targets.to(torch.int32).contiguous()
            out["action_logprobs"] = torch.empty(B, Tn, cfg.act_dim, dtype=torch.float32, device=self.device)
        so = L.XLSeqOutputs(tokens=out["action_tokens"].data_ptr(), actions=out["action_preds"].data_ptr(),
                            logits=_ptr(out.get("action_logits")).value, targets=_ptr(targets).value,
                            logprobs=_ptr(out.get("action_logprobs")).value)
        self._seq_call(state, states, rtg, rewards, lens, L.XL_FLAG_DISCRETE if discrete else 0, state_embeds, so)
        return out

    @_on_device
    def policy_step(self, state: StateCache, states: torch.Tensor, rtg: torch.Tensor,
                    rewards: Optional[torch.Tensor] = None, mode: int = L.XL_MODE_FUSED, flags: int = 0,
                    want_logits: bool = False, want_hidden: bool = False, out: Optional[dict] = None,
                    state_embeds: bool = False):
        """One env step of the policy. `states` [B, state_dim]; with `state_embeds=True` it is instead the
        state-token embedding [B, d] computed by the caller (image observations -> ImpalaCNN, or the reference's
        `img_is_encoded` inputs, discrete_decision_transformer_model.py:185-186) and embed_state is skipped."""
        cfg = self.cfg
        B = state.B
        if state_embeds:
            flags |= L.XL_FLAG_STATE_EMBEDS
        want = (B, cfg.d) if (flags & L.XL_FLAG_STATE_EMBEDS) else (B, cfg.state_dim)
        assert states.is_cuda and states.dtype == torch.float32 and tuple(states.shape) == want, \
            f"states must be a cuda fp32 tensor of shape {want}, got {tuple(states.shape)}"
        assert rtg.is_cuda and rtg.dtype == torch.float32 and rtg.numel() == B
        states, rtg = states.contiguous(), rtg.contiguous()
        if rewards is not None:
            rewards = rewards.to(self.device, torch.float32).contiguous()
        if out is None:
            out = {"action_tokens": torch.zeros(B, cfg.act_dim, dtype=torch.int32, device=self.device),
                   "action_preds": torch.zeros(B, cfg.act_dim, dtype=torch.float32, device=self.device)}
            if want_logits:
                n = cfg.num_actions if (flags & L.XL_FLAG_DISCRETE) else cfg.head_out
                out["action_logits"] = torch.empty(B, n, dtype=torch.float32, device=self.device)
            if want_hidden:
                out["last_hidden_state"] = torch.empty(B, cfg.tokens_per_step, cfg.d, dtype=torch.float32,
                                                       device=self.device)
        L.check(self.lib.xl_policy_step(
            self.handle, _ptr(state.buf), _ptr(states), _ptr(rtg), _ptr(rewards), _ptr(out["action_tokens"]),
            _ptr(out["action_preds"]), _ptr(out.get("action_logits")), _ptr(out.get("last_hidden_state")), B,
            mode, flags, self._stream()))
        return out

    @_on_device
    def policy_step_host(self, state: StateCache, h_states: torch.Tensor, h_rtg: torch.Tensor,
                         h_tokens: torch.Tensor, h_actions: torch.Tensor, mode: int = L.XL_MODE_FUSED,
                         flags: int = 0):
        """Host (pinned) buffers in, host buffers out; synchronises the stream. One env step end to end."""
        assert not h_states.is_cuda and not h_tokens.is_cuda
        L.check(self.lib.xl_policy_step_host(self.handle, _ptr(state.buf), _ptr(h_states), _ptr(h_rtg), _ptr(None),
                                             _ptr(h_tokens), _ptr(h_actions), state.B, mode, flags, self._stream()))

    @_on_device
    def cell_step(self, Cs, n, m, qkv, igate, fgate, outnorm_w, B: int, T: int, rows_split: int = 0,
                  cols_per_cta: int = 0, want_raw: bool = True, slab: bool = False):
        """Unit-parity entry point. `Cs` is given and updated in the REFERENCE layout [B,NH,DH,DH] unless
        `slab=True` (then it already is the library's slab-major layout and no conversion copies are made)."""
        inner = self.cfg.inner
        h_norm = torch.empty(B * T, inner, dtype=torch.float32, device=self.device)
        h_raw = torch.empty_like(h_norm) if want_raw else None
        Cp = Cs if slab else c_to_slab(Cs)
        L.check(self.lib.xl_mlstm_cell_step(self.handle, _ptr(Cp), _ptr(n), _ptr(m), _ptr(qkv), _ptr(igate),
                                            _ptr(fgate), _ptr(outnorm_w), _ptr(h_norm), _ptr(h_raw), B, T,
                                            rows_split, cols_per_cta, self._stream()))
        if not slab:
            Cs.copy_(c_from_slab(Cp))
        return h_norm, h_raw

    @_on_device
    def cell_seq(self, Cs, n, m, q, k, v, gates, act, u, outnorm_w, skip, B: int, S: int):
        """Unit-parity entry point of the sequence cell the "prefill_cell" option selects (xl_mlstm_cell_seq). `Cs` is
        given and updated in the REFERENCE layout [B,NH,DH,DH], n [B,NH,DH] and m [B,NH] in place. Returns
        (num [B*S, inner], qn [B*S, NH], m [B*NH, S], out [B*S, inner], cell id: 0 fp32, 1 mma.sync, 2 tcgen05)."""
        inner, NH = self.cfg.inner, self.cfg.num_heads
        num = torch.empty(B * S, inner, dtype=torch.float32, device=self.device)
        qn = torch.empty(B * S, NH, dtype=torch.float32, device=self.device)
        mseq = torch.empty(B * NH, S, dtype=torch.float32, device=self.device)
        out = torch.empty_like(num)
        cell = C.c_int(-1)
        Cp = c_to_slab(Cs)
        L.check(self.lib.xl_mlstm_cell_seq(self.handle, _ptr(Cp), _ptr(n), _ptr(m), _ptr(q), _ptr(k), _ptr(v),
                                           _ptr(gates), _ptr(act), _ptr(u), _ptr(outnorm_w), _ptr(skip), _ptr(num),
                                           _ptr(qn), _ptr(mseq), _ptr(out), C.addressof(cell), B, S, self._stream()))
        Cs.copy_(c_from_slab(Cp))
        return num, qn, mseq, out, cell.value

    @_on_device
    def linear(self, A: torch.Tensor, W_bf16: torch.Tensor, bias=None, residual=None, impl: int = 0):
        M, K = A.shape
        N = W_bf16.shape[0]
        assert W_bf16.dtype == torch.bfloat16 and W_bf16.shape[1] == K
        out = torch.empty(M, N, dtype=torch.float32, device=self.device)
        L.check(self.lib.xl_linear(self.handle, _ptr(A.contiguous()), _ptr(W_bf16.contiguous()), _ptr(bias),
                                   _ptr(residual), _ptr(out), M, N, K, impl, self._stream()))
        return out

    @_on_device
    def set_token_ring(self, ring: Optional[torch.Tensor], next_slot: int = 0):
        """Arm (or, `ring=None`, disarm) the token ring: int32 cuda tensor [slots, B, act_dim]; every policy step then
        also stores its action tokens in slot (steps since arming + next_slot) % slots. Same ring again = re-seek."""
        if ring is not None:
            assert ring.is_cuda and ring.dtype == torch.int32 and ring.is_contiguous() and ring.dim() == 3
            assert ring.shape[2] == self.cfg.act_dim
        self._token_ring = ring                       # keep it alive
        L.check(self.lib.xl_set_token_ring(self.handle, _ptr(ring), 0 if ring is None else ring.shape[0],
                                           int(next_slot), self._stream()))

    def set_sampling(self, temperature: Optional[float] = 1.0, top_k: int = 0, top_p: float = 0.5, seed: int = 0,
                     env_id_base: int = 0, env_id_stride: int = 1, step0: int = 0):
        """Arm the device sampler (`set_sampling(None)` disarms): every policy step then draws its action tokens by the
        `sample_from_logits` rule (defaults are its defaults) from a Philox stream keyed on (seed, step, global env id,
        action row) instead of taking the argmax; contract at xl_set_sampling in include/xlstm_b200.h. The first step
        after arming draws for step `step0`. Env b of this engine has global id env_id_base + b * env_id_stride (a shard
        of envs i -> rank i mod N: base = rank, stride = N). Parameters are checked before anything reaches the GPU."""
        p = None if temperature is None else sampling_params(self.cfg, temperature, top_k, top_p, seed, env_id_base,
                                                             env_id_stride)
        if not 0 <= int(step0) < 2 ** 32:
            raise ValueError(f"step0={step0} outside [0, 2^32)")
        with torch.cuda.device(self.device):
            L.check(self.lib.xl_set_sampling(self.handle, None if p is None else C.byref(p), int(step0), self._stream()))

    @_on_device
    def sample_actions(self, logits: torch.Tensor, step: int, temperature: float = 1.0, top_k: int = 0,
                       top_p: float = 0.5, seed: int = 0, env_id_base: int = 0, env_id_stride: int = 1,
                       discrete: bool = False):
        """The sampler alone on given logits (discrete [B, num_actions], continuous [B, act_dim * num_actions]) at an
        explicit step: -> (tokens int32 [B, act_dim], actions fp32 [B, act_dim]) as `policy_step` returns them
        (discrete: first column). Leaves the armed sampler alone."""
        cfg = self.cfg
        p = sampling_params(cfg, temperature, top_k, top_p, seed, env_id_base, env_id_stride)
        n = cfg.num_actions if discrete else cfg.head_out
        assert logits.is_cuda and logits.dtype == torch.float32 and logits.dim() == 2 and logits.shape[1] == n
        logits = logits.contiguous()
        B = logits.shape[0]
        tokens = torch.zeros(B, cfg.act_dim, dtype=torch.int32, device=self.device)
        actions = torch.zeros(B, cfg.act_dim, dtype=torch.float32, device=self.device)
        L.check(self.lib.xl_sample_actions(self.handle, _ptr(logits), B, L.XL_FLAG_DISCRETE if discrete else 0,
                                           C.byref(p), int(step) & 0xFFFFFFFF, _ptr(tokens), _ptr(actions),
                                           self._stream()))
        return tokens, actions

    @_on_device
    def set_option(self, name: str, value: int):
        L.check(self.lib.xl_set_option(self.handle, name.encode(), int(value)))

    def launch_count(self) -> int:
        return int(self.lib.xl_launch_count(self.handle))

    @_on_device
    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            torch.cuda.synchronize(self.device)
            self.lib.xl_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
