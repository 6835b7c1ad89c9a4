"""Batched rollout loop: the B-env restatement of `custom_evaluate_policy`
(src/callbacks/evaluation.py:14-271, which asserts num_envs == 1 at :80).

Per env, the reference's bookkeeping in inference-cache mode reduces to (SURVEY.md §3.1, App. C):
  * feed (state_t, rtg_t, reward placeholder 0) for the newest timestep only (:131-139, history pruned :172-177)
  * rtg_{t+1} = rtg_t - r_t / reward_scale                                       (:152-168)
  * on done: rtg <- target return, state history <- reset obs, past_key_values <- None (:238-251)
Here `past_key_values = None` for one env of the batch is a per-env reset mask handed to the library.

Multi-GPU: envs are sharded like the reference shards eval envs, `idx % world_size == rank`
(src/callbacks/custom_eval_callback.py:385,445); results go to every rank with ONE all_gather of the
action tokens / returns (the reference pickles dicts through gather_object, src/utils/misc.py:159-191).
"""
from __future__ import annotations

import time
import warnings
from typing import Any, Callable, Dict, List, Optional

import numpy as np
import torch

from . import _lib as L
from .engine import XLSTMEngine, check_lengths


def shard_env_ids(n_envs: int, rank: int, world_size: int) -> List[int]:
    """custom_eval_callback.py:385: env idx handled by rank idx % world_size."""
    return [i for i in range(n_envs) if i % world_size == rank]


def gather_env_results(local: torch.Tensor, n_envs: int, rank: int, world_size: int, group=None) -> torch.Tensor:
    """All-gather per-env rows (action tokens [B_local, A] or returns [B_local]) and put them back in global env
    order. One collective; works with NCCL (cuda tensors) and gloo (cpu tensors). Shards may be ragged."""
    import torch.distributed as dist
    if world_size == 1:
        return local
    max_local = (n_envs + world_size - 1) // world_size
    pad_shape = (max_local, *local.shape[1:])
    padded = torch.zeros(pad_shape, dtype=local.dtype, device=local.device)
    padded[: local.shape[0]] = local
    gathered = torch.empty((world_size, *pad_shape), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(gathered.view(-1, *local.shape[1:]), padded, group=group)
    out = torch.zeros((n_envs, *local.shape[1:]), dtype=local.dtype, device=local.device)
    for r in range(world_size):
        ids = shard_env_ids(n_envs, r, world_size)
        out[ids] = gathered[r, : len(ids)]
    return out


class OverlappedTokenGather:
    """All-gather of the action tokens, off the critical path and batched over `every` env steps.

    Step t's tokens are snapshotted into row t % every of one of two staging rings on the compute stream (a 2 KB
    copy); every `every` steps the ring is all-gathered on a side stream while the following steps compute. Envs
    never wait for other ranks' actions, so the only ordering needed is "ring k is not overwritten before its
    gather finished" (the gather of ring k overlaps the `every` steps that fill ring k ^ 1). `every = 1` is a
    gather per step; larger values amortise the collective's launch + SM footprint (the reference gathers
    results once, at the end of evaluation: src/utils/misc.py:159-191). `finish()` flushes a partly filled ring.
    Requires equal shards (B_local * world == n_envs). `results` collects, per flush, a [world, n_steps, B_local, A]
    tensor when `keep=True` (tests / callers that consume the gathered tokens); `global_view()` puts one step back
    in env order (env i lives on rank i % world). On CPU tensors (gloo) the same logic runs without streams.

    With `engine=` the two staging rings ARE the library's token ring (`xl_set_token_ring`): the argmax kernel at the
    end of every policy step writes the step's tokens into the ring slot itself (slot index advanced on the device,
    inside the captured graph), so `submit()` enqueues nothing between two graph replays — it only counts steps and
    launches the all-gather when a ring is full. Every policy step on that engine must then be followed by exactly
    one `submit()`.
    """

    def __init__(self, B_local: int, act_dim: int, world_size: int, device, group=None, every: int = 1,
                 keep: bool = False, engine=None):
        assert every >= 1
        self.world, self.group, self.every, self.keep = world_size, group, int(every), keep
        self.device = torch.device(device)
        self.cuda = self.device.type == "cuda"
        self.side = torch.cuda.Stream(device=self.device) if self.cuda else None
        mk = lambda *shape: torch.zeros(*shape, dtype=torch.int32, device=self.device)  # noqa: E731
        self.engine = engine
        if engine is not None:
            self.ring = mk(2 * self.every, B_local, act_dim)
            self.stage = [self.ring[: self.every], self.ring[self.every:]]
            engine.set_token_ring(self.ring, 0)
        else:
            self.stage = [mk(self.every, B_local, act_dim) for _ in range(2)]
        self.out = [mk(world_size, self.every, B_local, act_dim) for _ in range(2)]
        self.done = [None, None]
        self.k = 0            # ring being filled
        self.j = 0            # rows filled in ring k
        self.flushes = 0
        self.results: List[torch.Tensor] = []

    def submit(self, tokens: torch.Tensor) -> Optional[torch.Tensor]:
        """Queue one step's local tokens [B_local, A]. Returns the gathered [world, n, B_local, A] tensor of the
        flush this call triggered (valid on the compute stream after `finish()` or an event wait), else None."""
        k = self.k
        if self.engine is None:
            if self.cuda:
                cur = torch.cuda.current_stream(self.device)
                if self.j == 0 and self.done[k] is not None:
                    cur.wait_event(self.done[k])             # the previous gather of ring k still reads it
            self.stage[k][self.j].copy_(tokens, non_blocking=True)
        self.j += 1
        if self.j == self.every:
            return self._flush()
        return None

    def _flush(self) -> Optional[torch.Tensor]:
        import torch.distributed as dist
        k, n = self.k, self.j
        if n == 0:
            return None
        src = self.stage[k][:n]
        dst = self.out[k].view(-1)[: self.world * src.numel()].view(self.world, n, *src.shape[1:])
        if self.cuda:
            cur = torch.cuda.current_stream(self.device)
            ready = torch.cuda.Event()
            ready.record(cur)
            with torch.cuda.stream(self.side):
                self.side.wait_event(ready)
                dist.all_gather_into_tensor(dst.view(-1, src.shape[-1]), src.view(-1, src.shape[-1]),
                                            group=self.group)
                if self.keep:
                    self.results.append(dst.clone())
                ev = torch.cuda.Event()
                ev.record(self.side)
            self.done[k] = ev
        else:
            dist.all_gather_into_tensor(dst.view(-1, src.shape[-1]), src.reshape(-1, src.shape[-1]),
                                        group=self.group)
            if self.keep:
                self.results.append(dst.clone())
        self.flushes += 1
        self.k ^= 1
        self.j = 0
        if self.engine is not None:
            if self.cuda and self.done[self.k] is not None:
                # the next step writes into ring self.k: its previous gather must have finished reading it
                torch.cuda.current_stream(self.device).wait_event(self.done[self.k])
            if n != self.every:
                self.engine.set_token_ring(self.ring, self.k * self.every)   # partial flush: re-seek the device slot
        return dst

    def finish(self):
        """Flush a partly filled ring and make the compute stream wait for every outstanding gather."""
        self._flush()
        if self.cuda:
            for ev in self.done:
                if ev is not None:
                    torch.cuda.current_stream(self.device).wait_event(ev)

    def global_view(self, gathered: torch.Tensor) -> torch.Tensor:
        # [world, B_local, A] -> [n_envs, A]  (or [world, n, B_local, A] -> [n, n_envs, A]) with env = b * world + r
        if gathered.dim() == 4:
            return gathered.permute(1, 2, 0, 3).reshape(gathered.shape[1], -1, gathered.shape[-1])
        return gathered.permute(1, 0, 2).reshape(-1, gathered.shape[-1])


class BatchedRollout:
    """Drives B envs of a `SyntheticEnvBatch`-like object (reset() -> obs[B,204]; step(a) -> obs, reward, done)
    through the CUDA policy, one library call per env step with pinned host buffers.

    `sample_kwargs` (the reference's `a_sample_kwargs`: temperature, top_k, top_p; env_id_base / env_id_stride for a
    shard of a multi-GPU run) arms the engine's device sampler, so a sampled rollout is still one call per step. Draws
    come from a counter-based stream keyed on `seed` (None: one drawn from torch's global RNG); every `run()` without
    `keep_state` restarts it at step 0, so equal seeds give equal rollouts. The engine stays armed afterwards."""

    def __init__(self, engine: XLSTMEngine, envs, mode: int = L.XL_MODE_FUSED, use_graph: bool = True,
                 sample_kwargs: Optional[Dict[str, Any]] = None, seed: Optional[int] = None):
        self.engine, self.envs = engine, envs
        self.sample_kwargs = dict(sample_kwargs) if sample_kwargs is not None else None
        if self.sample_kwargs is not None:
            self.seed = int(torch.randint(0, 2 ** 62, ()).item()) if seed is None else int(seed)
            engine.set_sampling(**self.sample_kwargs, seed=self.seed, step0=0)
        self.B = envs.B
        cfg = engine.cfg
        self.mode = mode
        self.flags = L.XL_FLAG_GRAPH if use_graph else 0
        self.state = engine.new_state(self.B)
        pin = dict(pin_memory=True)
        self.h_states = torch.zeros(self.B, cfg.state_dim, dtype=torch.float32, **pin)
        self.h_rtg = torch.zeros(self.B, dtype=torch.float32, **pin)
        self.h_tokens = torch.zeros(self.B, cfg.act_dim, dtype=torch.int32, **pin)
        self.h_actions = torch.zeros(self.B, cfg.act_dim, dtype=torch.float32, **pin)
        self.rtg0 = np.asarray(envs.rtg0, dtype=np.float32)
        self.scale = np.asarray(envs.reward_scale, dtype=np.float32)

    def prefill_context(self, states, rtg, rewards=None, lengths=None) -> None:
        """Warm the recurrent state with a context of earlier timesteps before the rollout starts — the batched
        counterpart of `persist_context` (src/callbacks/evaluation.py:213-237), where the reference keeps the previous
        episodes' tokens in front of the new episode: states [B, Tn, state_dim], rtg [B, Tn], rewards [B, Tn] or None
        (the 0 placeholder the rollout feeds). Follow with `run(..., keep_state=True)`.

        lengths=None: every env is reset and takes all Tn timesteps; one chunkwise-parallel pass (`xl_policy_prefill`)
        leaves the state exactly where Tn recurrent env steps would. lengths (B ints in [0, Tn]; histories of different
        lengths, e.g. episodes that ended at different times): only the envs with lengths[b] > 0 are reset, each then
        takes its own first lengths[b] timesteps (`xl_policy_prefill_ragged`); envs with 0 keep their state, so a few
        envs of a running batch can be re-primed without touching the others."""
        lens = None
        if lengths is not None:
            Tn = (states.shape if hasattr(states, "shape") else np.shape(states))[1]
            lens = check_lengths(lengths, self.B, Tn, "Tn")
        dev = self.engine.device
        to = lambda a: None if a is None else torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32).to(dev)  # noqa: E731
        if lens is None:
            self.engine.reset(self.state)
        else:
            self.engine.reset(self.state, torch.from_numpy((lens > 0).astype(np.uint8)))
        self.engine.policy_prefill(self.state, to(states), to(rtg), to(rewards), lengths=lens)

    def run(self, n_steps: int, record: bool = False, keep_state: bool = False) -> Dict[str, object]:
        envs, B = self.envs, self.B
        obs = envs.reset()
        rtg = self.rtg0.copy()
        if not keep_state:
            self.engine.reset(self.state)
            if self.sample_kwargs is not None:
                self.engine.set_sampling(**self.sample_kwargs, seed=self.seed, step0=0)
        ep_ret = np.zeros(B, dtype=np.float64)
        returns: List[List[float]] = [[] for _ in range(B)]
        toks = [] if record else None
        acts = [] if record else None
        t0 = time.perf_counter()
        for _ in range(n_steps):
            self.h_states.numpy()[:] = obs
            self.h_rtg.numpy()[:] = rtg
            self.engine.policy_step_host(self.state, self.h_states, self.h_rtg, self.h_tokens, self.h_actions,
                                         mode=self.mode, flags=self.flags)
            actions = self.h_actions.numpy()
            if record:
                toks.append(self.h_tokens.numpy().copy())
                acts.append(actions.copy())
            # env_act_dim truncation (discrete_decision_transformer_sb3.py:70-71) is per env
            obs, reward, done = envs.step(actions)
            ep_ret += reward
            rtg = (rtg - reward / self.scale).astype(np.float32)
            if done.any():
                for i in np.nonzero(done)[0]:
                    returns[i].append(float(ep_ret[i]))
                    ep_ret[i] = 0.0
                rtg[done] = self.rtg0[done]
                self.engine.reset(self.state, torch.from_numpy(done.astype(np.uint8)))
        dt = time.perf_counter() - t0
        out: Dict[str, object] = {
            "env_steps": n_steps * B, "seconds": dt,
            # the reference's metric names (custom_eval_callback.py:468-475)
            "steps_per_second": n_steps / dt, "total_steps_per_second": n_steps * B / dt,
            "episode_returns": returns,
        }
        if record:
            out["tokens"] = np.stack(toks)
            out["actions"] = np.stack(acts)
        return out


def _action_dim(space) -> int:
    """stable_baselines3.common.preprocessing.get_action_dim for Box / Discrete spaces."""
    if hasattr(space, "n"):
        return 1
    return int(np.prod(space.shape))


def custom_evaluate_policy(model, env, n_eval_episodes: int = 10, deterministic: bool = True, render: bool = False,
                           callback: Optional[Callable[[Dict[str, Any], Dict[str, Any]], None]] = None,
                           reward_threshold: Optional[float] = None, return_episode_rewards: bool = False,
                           warn: bool = True, task_id: int = 0):
    """`custom_evaluate_policy` (src/callbacks/evaluation.py:14-271) with the reference's signature and return values,
    for `env.num_envs >= 1` (the reference asserts == 1 at :80): all envs of the VecEnv step through ONE batched policy
    call per env step, each env keeping its own recurrent state in the agent's `past_key_values` (a `StateCache`).

    `model` is the agent (`lram_b200.decision_xlstm.DiscreteDecisionXLSTM`): the loop reads `model.policy`,
    `model.device`, `model.compute_target_return_val`, `model.get_reward_scale_for_env`, `model.persist_context`,
    `model.past_key_values`, exactly the attributes the reference loop reads. Per env, in inference-cache mode:
      * the policy sees (state_t, rtg_t, reward placeholder 0) of the newest timestep (:130-139, 172-177),
      * rtg_{t+1} = rtg_t - r_t / reward_scale in fp32 (:152-168),
      * on done: rtg <- target return; the recurrent state is reset (`past_key_values = None`, :238-251) UNLESS
        `model.persist_context` (:213-237), where the context — here the recurrent state — carries over episodes,
      * `model.reset_inf_cache_freq` (decision_transformer_sb3.py:663-666): an env's state is also dropped after the
        prediction at every timestep t > 0 with t % freq == 0,
      * episodes are divided among the envs as SB3 does (:87-89); episode reward / length bookkeeping follows
        :199-211 (Monitor `info["episode"]` when present; otherwise the reference appends the LAST step's reward).
    """
    n_envs = int(env.num_envs)
    action_dim = _action_dim(env.action_space)
    discrete_env = hasattr(env.action_space, "n")
    if warn and not getattr(env, "is_monitor_wrapped", False):
        warnings.warn("Evaluation environment is not wrapped with a ``Monitor`` wrapper.", UserWarning)
    episode_rewards, episode_lengths, episode_times = [], [], []
    episode_counts = np.zeros(n_envs, dtype="int")
    episode_count_targets = np.array([(n_eval_episodes + i) // n_envs for i in range(n_envs)], dtype="int")
    current_rewards = np.zeros(n_envs)
    current_lengths = np.zeros(n_envs, dtype="int")
    observations = np.asarray(env.reset())
    target = np.float32(model.compute_target_return_val(env=env, task_id=task_id))
    rtg = np.full(n_envs, target, dtype=np.float32)
    env_name = getattr(getattr(env, "envs", [None])[0], "name", None)
    reward_scale = np.float32(model.get_reward_scale_for_env(envid=env_name))
    model.past_key_values = None                                   # :120-124
    persist = bool(getattr(model, "persist_context", False))
    reset_freq = getattr(model, "reset_inf_cache_freq", None)
    timestep = np.zeros(n_envs, dtype="int")                         # per-env `timesteps[0, -1]` of the reference loop
    start_time = [time.time()] * n_envs
    while (episode_counts < episode_count_targets).any():
        obs_t = torch.from_numpy(observations)
        actions = model.predict_batch(model.policy, obs_t, torch.from_numpy(rtg), action_dim,
                                      env_act_dim=action_dim)
        a_np = actions.detach().cpu().numpy()
        if discrete_env:
            a_np = a_np.astype(int).reshape(n_envs)                # :142-143
        observations, reward, done, infos = env.step(a_np if n_envs > 1 or discrete_env else [a_np[0]])
        observations = np.asarray(observations)
        reward = np.asarray(reward)
        done = np.asarray(done).astype(bool).reshape(n_envs)
        current_rewards += reward
        current_lengths += 1
        rtg = np.where(done, target, rtg - reward.astype(np.float32) / reward_scale).astype(np.float32)
        for i in range(n_envs):
            if episode_counts[i] < episode_count_targets[i]:
                info = infos[i] if infos is not None else {}
                if callback is not None:
                    callback(locals(), globals())
                if done[i]:
                    episode_times.append(time.time() - start_time[i])
                    start_time[i] = time.time()
                    if "episode" in info:
                        episode_rewards.append(info["episode"]["r"])
                        episode_lengths.append(info["episode"]["l"])
                    else:
                        episode_rewards.append(reward[i:i + 1] if n_envs > 1 else reward)   # :208 (sic)
                        episode_lengths.append(current_lengths[i] if n_envs > 1 else current_lengths[0])
                    episode_counts[i] += 1
        drop = done & (not persist)
        if reset_freq is not None:
            drop = drop | ((timestep > 0) & (timestep % int(reset_freq) == 0))
        timestep = np.where(done, 0, timestep + 1)
        if drop.any() and model.past_key_values is not None:
            cache = model.past_key_values
            cache.engine.reset(cache, torch.from_numpy(drop.astype(np.uint8)))
        if render:
            env.render()
    model.past_key_values = None                                   # :259-262
    mean_reward, std_reward = np.mean(episode_rewards), np.std(episode_rewards)
    if reward_threshold is not None:
        assert mean_reward > reward_threshold, f"Mean reward below threshold: {mean_reward:.2f} < {reward_threshold:.2f}"
    if return_episode_rewards:
        return episode_rewards, episode_lengths, episode_times
    return mean_reward, std_reward, np.mean(episode_times)
