"""Image front-end of the policy: `embed_image` = IMPALA CNN (SURVEY.md §8 a12).

Reference: `ImpalaCNN` / `ImpalaCNNBlock` / `ImpalaCNNResidual` (src/algos/models/image_encoders.py:10-125), built by
`make_image_encoder` for `image_shape=[3,64,64]` (multi_domain_discrete_dt_model.py:38-46,
configs/agent_params/model_kwargs/multi_domain.yaml) and applied to `states.float() / 255`
(online_decision_transformer_model.py:522-526) one timestep at a time on the rollout path
(discrete_decision_transformer_model.py:187-203).

Per SURVEY.md §8 a12 this stage stays in PyTorch / cuDNN (it is not on the HBM-bound recurrent path): three
stages of conv3x3 -> maxpool(3, stride 2, pad 1) -> 2 residual units (relu -> conv3x3 -> relu -> conv3x3, skip),
channels 16/32/32 x model_size, then ReLU, flatten, Linear(n_flat -> d), ReLU. Parameter names equal the
reference's, so `embed_image.*` entries of an LRAM checkpoint load with `load_state_dict`. The resulting state
embeddings [B, d] enter the CUDA path through `xl_policy_step(..., XL_FLAG_STATE_EMBEDS)`; whole trajectories
([B, T, d] from `embed_frames`) through `xl_policy_prefill_embeds` / `xl_policy_forward_embeds`.
(Spectral-norm and modulation-vector variants of the reference class are training options, unused by the
multi_domain configuration, and are not reproduced.)
"""
from __future__ import annotations

from typing import Dict, Sequence

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F


class _Residual(nn.Module):
    def __init__(self, depth: int):
        super().__init__()
        self.conv_0 = nn.Conv2d(depth, depth, 3, 1, 1)
        self.conv_1 = nn.Conv2d(depth, depth, 3, 1, 1)

    def forward(self, x):
        y = self.conv_0(F.relu(x))
        y = self.conv_1(F.relu(y))
        return x + y


class _Stage(nn.Module):
    def __init__(self, depth_in: int, depth_out: int):
        super().__init__()
        self.conv = nn.Conv2d(depth_in, depth_out, 3, 1, 1)
        self.residual_0 = _Residual(depth_out)
        self.residual_1 = _Residual(depth_out)

    def forward(self, x):
        x = F.max_pool2d(self.conv(x), 3, 2, padding=1)
        return self.residual_1(self.residual_0(x))


class ImpalaCNN(nn.Module):
    def __init__(self, image_shape: Sequence[int] = (3, 64, 64), features_dim: int = 512, model_size: int = 1,
                 out_relu: bool = True):
        super().__init__()
        c, hgt, wid = image_shape
        self.image_shape = tuple(image_shape)
        self.cnn = nn.ModuleList([_Stage(c, 16 * model_size), _Stage(16 * model_size, 32 * model_size),
                                  _Stage(32 * model_size, 32 * model_size)])
        for _ in range(3):                                   # maxpool(3, 2, pad 1): n -> floor((n - 1) / 2) + 1
            hgt, wid = (hgt - 1) // 2 + 1, (wid - 1) // 2 + 1
        self.n_flatten = 32 * model_size * hgt * wid
        self.linear = nn.Sequential(nn.Linear(self.n_flatten, features_dim), nn.ReLU() if out_relu else nn.Identity())

    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x [N, C, H, W] float, ALREADY scaled to 0..1: the caller divides raw frames by 255 exactly once, as the
        reference's `embed_inputs` does before `embed_image` (online_decision_transformer_model.py:522-526)."""
        if not x.is_floating_point():
            raise TypeError("ImpalaCNN takes float frames already scaled by 1/255 (see scale_frames)")
        for stage in self.cnn:
            x = stage(x)
        return self.linear(torch.flatten(F.relu(x), 1))


def scale_frames(frames: torch.Tensor) -> torch.Tensor:
    """`states.float() / 255.0` (online_decision_transformer_model.py:523-525), unconditionally: image observations
    reach the policy as raw 0..255 values whether their dtype is uint8 or — after `pad_inputs` returned
    `states.float()` (src/algos/decision_xlstm.py:25) — float."""
    return frames.float() / 255.0


@torch.no_grad()
def embed_frames(cnn: ImpalaCNN, frames: torch.Tensor, lengths=None, max_frames: int = 2048) -> torch.Tensor:
    """State embeddings of whole trajectories of raw frames, the input of the sequence calls with `state_embeds=True`
    (`XLSTMEngine.policy_forward` / `policy_prefill`): frames [B, T, C, H, W], uint8 or float with values 0..255, on
    any device -> fp32 [B, T, d] on the CNN's device. `scale_frames` is applied once per frame, and the CNN runs on at
    most `max_frames` frames at a time (at T in the tens of thousands one batch of first-stage activations would not
    fit). `lengths` (B ints in [0, T]): frames at or past lengths[b] are never fed to the CNN and their rows are 0."""
    if not isinstance(frames, torch.Tensor) or frames.dim() != 5:
        raise ValueError(f"frames must be a [B, T, C, H, W] tensor, got {getattr(frames, 'shape', type(frames))}")
    if tuple(frames.shape[2:]) != tuple(cnn.image_shape):
        raise ValueError(f"frames must be [B, T, {', '.join(map(str, cnn.image_shape))}], got {tuple(frames.shape)}")
    if max_frames < 1:
        raise ValueError(f"max_frames={max_frames} must be positive")
    B, T = frames.shape[:2]
    dev = cnn.linear[0].weight.device
    out = torch.zeros(B, T, cnn.linear[0].out_features, dtype=torch.float32, device=dev)
    flat, out_flat = frames.reshape(B * T, *frames.shape[2:]), out.view(B * T, -1)
    if lengths is None:
        for i in range(0, B * T, max_frames):
            out_flat[i:i + max_frames] = cnn(scale_frames(flat[i:i + max_frames].to(dev)))
        return out
    from .engine import check_lengths
    lens = torch.from_numpy(check_lengths(lengths, B, T, "T").astype(np.int64))
    rows = (torch.arange(T).view(1, T) < lens.view(B, 1)).view(-1).nonzero().view(-1)   # valid frames, in order
    for i in range(0, rows.numel(), max_frames):
        idx = rows[i:i + max_frames]
        x = flat.index_select(0, idx.to(flat.device))
        out_flat.index_copy_(0, idx.to(dev), cnn(scale_frames(x.to(dev))))
    return out


def make_impala_state_dict(features_dim: int, image_shape: Sequence[int] = (3, 64, 64), seed: int = 0,
                           prefix: str = "embed_image.") -> Dict[str, torch.Tensor]:
    """Seeded default-init weights with the reference's key names (for synthetic policies and tests)."""
    g = torch.Generator().manual_seed(seed)
    with torch.random.fork_rng():
        torch.manual_seed(int(torch.randint(0, 2 ** 31 - 1, (1,), generator=g)))
        net = ImpalaCNN(image_shape, features_dim)
    return {prefix + k: v.detach().clone() for k, v in net.state_dict().items()}


def split_image_weights(sd: Dict[str, torch.Tensor], prefix: str = "embed_image.") -> Dict[str, torch.Tensor]:
    return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}
