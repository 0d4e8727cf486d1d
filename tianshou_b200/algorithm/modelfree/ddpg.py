"""DDPG with the whole ``update()`` on the device, and the off-policy actor-critic base that DDPG, TD3 and SAC share.

Reference: tianshou/algorithm/modelfree/ddpg.py (ContinuousPolicyWithExplorationNoise :41-111, ContinuousDeterministicPolicy
:114-190, ActorCriticOffPolicyAlgorithm :196-339, DDPG :342-410), utils/net/continuous.py:32-85 (deterministic actor),
utils/lagged_network.py:8-80 (Polyak).

Per ``update(buffer, sample_size)`` of DDPG:
  host : index draw (``buffer.sample_indices``: the reference's numpy RandomState streams), one D2H of the loss scalars.
  GPU  : row gathers from the buffer's device mirror (or one upload of the sampled rows), lagged actor forward ->
         ``ts_det_actor_head`` -> lagged critic -> ``ts_nstep_return``; critic forward / ``ts_critic_mse`` / backward + Adam;
         actor forward, critic input-gradient GEMMs, ``ts_det_actor_head_bwd``, actor backward + Adam; Polyak on every
         lagged network.
Every Linear layer's forward / input gradient / weight gradient is one tcgen05 GEMM launch (csrc/net_gemm.cu).
"""
from __future__ import annotations

import time
import warnings
from collections.abc import Hashable
from copy import deepcopy
from dataclasses import dataclass
from typing import Any, Literal

import numpy as np
import torch
from torch import nn

from ..._cabi import call, ptr, stream_ptr, to_device
from ...data import Batch, ReplayBuffer
from ...exploration import BaseNoise, GaussianNoise
from ..base import OffPolicyAlgorithm, Policy, TrainingStats, _space_kind
from ..flat_params import UnsupportedModelError
from ..netgraph import ACT_NONE, FlatGroup, FusedStack, _Layer, compile_sequential, module_layers, polyak_update
from ..optim import OptimizerFactory


@dataclass(kw_only=True)
class DDPGTrainingStats(TrainingStats):
    actor_loss: float
    critic_loss: float


class ContinuousDeterministicPolicy(Policy):
    """s -> action policy of DDPG / TD3 (ddpg.py:41-190).  ``forward`` is the torch-module path the Collector runs."""

    def __init__(self, *, actor: nn.Module, exploration_noise: BaseNoise | Literal["default"] | None = None, action_space: Any,
                 observation_space: Any | None = None, action_scaling: bool = True,
                 action_bound_method: Literal["clip"] | None = "clip") -> None:
        if action_scaling and not np.isclose(actor.max_action, 1.0):
            warnings.warn("action_scaling and action_bound_method are only intended to deal with unbounded model action space, "
                          f"but find actor model bound action space with max_action={actor.max_action}. Consider using "
                          "unbounded=True option of the actor model, or set action_scaling to False and action_bound_method to None.")
        super().__init__(action_space=action_space, observation_space=observation_space, action_scaling=action_scaling,
                         action_bound_method=action_bound_method)
        if exploration_noise == "default":
            exploration_noise = GaussianNoise(sigma=0.1)
        self.exploration_noise = exploration_noise
        self.actor = actor

    def set_exploration_noise(self, noise: BaseNoise | None) -> None:
        self.exploration_noise = noise

    def add_exploration_noise(self, act: Any, batch: Any) -> Any:
        if self.exploration_noise is None:
            return act
        if isinstance(act, np.ndarray):
            return act + self.exploration_noise(act.shape)
        warnings.warn("Cannot add exploration noise to non-numpy_array action.")
        return act

    def forward(self, batch: Batch, state: Any = None, model: nn.Module | None = None, **kwargs: Any) -> Batch:
        actions, hidden = (model or self.actor)(batch.obs, state=state, info=batch.get("info"))
        return Batch(act=actions, state=hidden)


# ------------------------------------------------------------------------------------------------ module -> kernel views
def _linear_relu_chain(mod: Any, in_dim: int, what: str) -> list[_Layer]:
    try:
        return compile_sequential(module_layers(mod), (in_dim,))
    except UnsupportedModelError as e:
        raise UnsupportedModelError(f"{what}: {e}") from e


def _chain_params(layers: list[_Layer]) -> list[nn.Parameter]:
    params: list[nn.Parameter] = []
    for L in layers:
        params += [L.weight, L.bias]
    return params


def describe_q_critic(critic: Any, obs_dim: int, act_dim: int) -> tuple[list[_Layer], list[nn.Parameter]]:
    """ContinuousCritic(preprocess_net=Net(concat=True), ...) -> Linear/ReLU chain on concat(obs, act) ending in 1 output."""
    if getattr(critic, "apply_preprocess_net_to_obs_only", False):
        raise UnsupportedModelError("critic: apply_preprocess_net_to_obs_only unsupported")
    layers = _linear_relu_chain(critic.preprocess, obs_dim + act_dim, "critic.preprocess")
    if getattr(critic.preprocess, "softmax", False):
        raise UnsupportedModelError("critic: softmax trunk output unsupported")
    layers += _linear_relu_chain(critic.last, layers[-1].out_dim, "critic.last")
    if layers[-1].out_dim != 1 or layers[-1].act != ACT_NONE:
        raise UnsupportedModelError("critic must end in a single linear Q output")
    return layers, _chain_params(layers)


def describe_deterministic_actor(actor: Any, obs_dim: int) -> tuple[list[_Layer], list[nn.Parameter], int]:
    """ContinuousActorDeterministic: preprocess + ``last`` chain ending in a linear [A, H] layer; ``max_action * tanh`` is the
    head kernel.  Parameters in ``actor.parameters()`` order."""
    layers = _linear_relu_chain(actor.preprocess, obs_dim, "actor.preprocess")
    layers += _linear_relu_chain(actor.last, layers[-1].out_dim, "actor.last")
    if layers[-1].act != ACT_NONE:
        raise UnsupportedModelError("actor.last must end in a linear layer (max_action * tanh is applied by the actor)")
    return layers, _chain_params(layers), layers[-1].out_dim


class ActorCriticOffPolicyAlgorithm(OffPolicyAlgorithm):
    """Actor + critic(s) with lagged copies, n-step critic targets and Polyak updates (ddpg.py:196-339), on the device.

    Holds what DDPG, TD3 and SAC share: the fused actor / critic stacks and their flat parameter groups, the row gathers,
    the critic step, Polyak on every lagged network, and the CUDA-graph mode of ``update()``.  Subclasses define the actor
    head, the target value and ``_update_with_batch``."""

    _n_noise = 0        # standard-normal [B, A] draws of one update (persistent inputs of the graphed body)
    _n_losses = 2       # loss scalars read back after one update

    def __init__(self, *, policy: Policy, policy_optim: OptimizerFactory, critic: nn.Module, critic_optim: OptimizerFactory,
                 tau: float = 0.005, gamma: float = 0.99, n_step_return_horizon: int = 1, cuda_graph: bool = False) -> None:
        assert 0.0 <= tau <= 1.0, f"tau should be in [0, 1] but got: {tau}"
        assert 0.0 <= gamma <= 1.0, f"gamma should be in [0, 1] but got: {gamma}"
        super().__init__(policy=policy)
        if _space_kind(policy.action_space) != "continuous":
            raise ValueError(f"{type(policy).__name__} only supports Box action spaces, but got {policy.action_space=}.")
        self.tau = tau
        self.gamma = gamma
        self.n_step_return_horizon = n_step_return_horizon
        dev = next(policy.actor.parameters()).device
        if dev.type != "cuda":
            raise UnsupportedModelError(f"networks live on {dev}; tianshou_b200 has no CPU path -- move them to a CUDA device")
        self._dev = dev
        self.obs_dim = int(module_layers(policy.actor.preprocess)[0].in_features)
        a_layers, a_params, self.act_dim = self._describe_actor(policy.actor)
        self._g_actor = FlatGroup(a_params, dev)
        self._actor = FusedStack(a_layers, self._g_actor, "actor")
        self._g_c: list[FlatGroup] = []
        self._c: list[FusedStack] = []
        self._g_ct: list[FlatGroup] = []
        self._lagged: list[tuple[FlatGroup, FlatGroup]] = []       # (target, source) pairs of the Polyak update
        self._g_at: FlatGroup | None = None
        self.policy_optim = self._fused_optimizer(policy, policy_optim, self._g_actor)
        self.critic = critic
        self.critic_old = self._add_critic(critic)
        self.critic_optim = self._fused_optimizer(critic, critic_optim, self._g_c[0])
        self._scratch: dict[str, torch.Tensor] = {}
        # opt-in: the device work of one update() captured once into a CUDA graph and replayed -- the eager call sequence is
        # Python-launch bound.  Needs a buffer with a device mirror and uniform replay.
        self.cuda_graph = bool(cuda_graph)
        self._graphs: dict[Hashable, dict[str, Any]] = {}     # one graph per control-flow variant of the update
        self._graph: dict[str, Any] = {}                      # the variant the last update ran
        self._adam = FlatGroup.adam_step          # the graphed body switches to the device-step variant
        # standard-normal noise source: torch's generator on the networks' device (what the reference draws when it runs there)
        self._noise_fn = lambda shape: torch.normal(torch.zeros(shape, device=dev), torch.ones(shape, device=dev))

    # ------------------------------------------------------------------ construction helpers
    def _describe_actor(self, actor: nn.Module) -> tuple[list[_Layer], list[nn.Parameter], int]:
        return describe_deterministic_actor(actor, self.obs_dim)

    def _add_critic(self, critic: nn.Module) -> nn.Module:
        """Fuse ``critic`` and return its lagged copy (a plain deepcopy, Polyak-updated on the device)."""
        critic_old = deepcopy(critic).eval()
        layers, params = describe_q_critic(critic, self.obs_dim, self.act_dim)
        _, tparams = describe_q_critic(critic_old, self.obs_dim, self.act_dim)
        g = FlatGroup(params, self._dev)
        self._g_c.append(g)
        self._c.append(FusedStack(layers, g, "critic"))
        self._g_ct.append(FlatGroup(tparams, self._dev))
        self._lagged.append((self._g_ct[-1], g))
        return critic_old

    def _add_lagged_actor(self) -> None:
        """``actor_old``: the lagged actor that computes the target action (ddpg.py:398, td3.py:183)."""
        self.actor_old = deepcopy(self.policy.actor).eval()
        _, tparams, _ = self._describe_actor(self.actor_old)
        self._g_at = FlatGroup(tparams, self._dev)
        self._lagged.append((self._g_at, self._g_actor))

    def _fused_optimizer(self, module: nn.Module, factory: OptimizerFactory, group: FlatGroup) -> Any:
        optim = self._create_optimizer(module, factory)
        if set(map(id, optim._optim.param_groups[0]["params"])) != set(map(id, group.params)):
            raise UnsupportedModelError("optimizer parameters differ from the fused network's parameters")
        optim._flat = group
        return optim

    # ------------------------------------------------------------------ helpers
    def _buf(self, name: str, shape: tuple[int, ...] | int, dtype: torch.dtype = torch.float32) -> torch.Tensor:
        shape = (shape,) if isinstance(shape, int) else tuple(shape)
        t = self._scratch.get(name)
        if t is None or t.shape != shape or t.dtype != dtype:
            t = self._scratch[name] = torch.empty(shape, dtype=dtype, device=self._dev)
        return t

    def _rows(self, buffer: ReplayBuffer, key: str, indices: np.ndarray | torch.Tensor) -> torch.Tensor:
        """buffer[key][indices] as a dense fp32 [I, width] device tensor: gathered from the device mirror when the
        buffer keeps one (no host traffic), else a host gather of the sampled rows + one upload."""
        cols = self._cols_override if self._cols_override is not None else (
            buffer.device_columns() if hasattr(buffer, "device_columns") else None)
        if cols is not None and key in cols:
            from ... import ops
            idx = indices if isinstance(indices, torch.Tensor) else to_device(np.asarray(indices, dtype=np.int64), self._dev)
            src = cols[key]
            return ops.gather_rows(src.reshape(src.shape[0], -1), idx).to(torch.float32)
        arr = np.asarray(buffer._meta[key])[np.asarray(indices)]
        return to_device(np.ascontiguousarray(arr.reshape(len(arr), -1)), self._dev, dtype=torch.float32)

    def _obs_next(self, buffer: ReplayBuffer, indices: np.ndarray | torch.Tensor) -> torch.Tensor:
        if buffer._save_obs_next:
            return self._rows(buffer, "obs_next", indices).contiguous()
        return self._rows(buffer, "obs", buffer.next(indices)).contiguous()

    def _q_forward(self, k: int, obs: torch.Tensor, act: torch.Tensor, tag: str, target: bool = False) -> tuple[list[torch.Tensor], torch.Tensor]:
        B = obs.shape[0]
        x = self._buf(f"{tag}_x{k}", (B, self.obs_dim + self.act_dim))
        call("ts_concat2", ptr(obs), self.obs_dim, ptr(act), self.act_dim, B, ptr(x), stream_ptr(self._dev))
        if target:
            self._g_ct[k].ensure_adopted()
        acts = self._c[k].forward(x, B, tag, params=self._g_ct[k].flat if target else None)
        return acts, acts[-1].view(B)

    @property
    def _max_action(self) -> float:
        return float(self.policy.actor.max_action)

    # ------------------------------------------------------------------ target
    def _target_smoothing(self, B: int) -> tuple[torch.Tensor | None, float, float]:
        """(noise, policy_noise, noise_clip) of target-policy smoothing; DDPG has none and draws nothing."""
        return None, 0.0, 0.0

    def _target_q_compute_value(self, obs_next: torch.Tensor, act: torch.Tensor) -> torch.Tensor:
        """critic_old(s', a')  (ddpg.py:314-325)"""
        acts, _ = self._q_forward(0, obs_next, act, "tq", target=True)
        return acts[-1]

    def _target_q(self, buffer: ReplayBuffer, indices: np.ndarray) -> torch.Tensor:
        """Q'(s', actor_old(s') [+ smoothing noise])   (ddpg.py:327-339, 400-402, td3.py:190-202)"""
        obs_next = self._obs_next(buffer, indices)
        B, A = obs_next.shape[0], self.act_dim
        self._g_at.ensure_adopted()
        z = self._actor.forward(obs_next, B, "tq", params=self._g_at.flat)[-1]
        noise, policy_noise, noise_clip = self._target_smoothing(B)
        act = self._buf("tq_act", (B, A))
        call("ts_det_actor_head", ptr(z), A, B, A, self._max_action, ptr(noise), policy_noise, noise_clip, ptr(act),
             stream_ptr(self._dev))
        return self._target_q_compute_value(obs_next, act)

    def _preprocess_batch(self, batch: Batch, buffer: ReplayBuffer, indices: np.ndarray) -> Batch:
        return self.compute_nstep_return(batch=batch, buffer=buffer, indices=indices, target_q_fn=self._target_q,
                                         gamma=self.gamma, n_step=self.n_step_return_horizon)

    def _sample(self, buffer: ReplayBuffer, sample_size: int | None) -> tuple[Batch, Any]:
        """Indices from the buffer's host RNG streams (identical to the reference's draws); rows stay on the device."""
        indices = buffer.sample_indices(sample_size)
        batch = Batch()
        batch.__dict__["obs"] = self._rows(buffer, "obs", indices).contiguous()
        batch.__dict__["act"] = self._rows(buffer, "act", indices).contiguous()
        if hasattr(buffer, "get_weight"):          # PrioritizedReplayBuffer.__getitem__ adds the IS weight (prio.py:104-106)
            w = buffer.get_weight(indices)
            batch.__dict__["weight"] = to_device(np.asarray(w / np.max(w) if buffer._weight_norm else w, dtype=np.float32), self._dev)
        batch.__dict__["info"] = Batch()
        return batch, indices

    # ------------------------------------------------------------------ update pieces
    def _returns_and_weight(self, batch: Batch) -> tuple[torch.Tensor, torch.Tensor | None]:
        returns = batch.returns.reshape(-1).to(self._dev, torch.float32).contiguous()
        weight = getattr(batch, "weight", None)
        if weight is not None and not isinstance(weight, torch.Tensor):
            weight = to_device(np.asarray(weight, dtype=np.float32), self._dev)
        if weight is not None:
            weight = weight.reshape(-1).to(self._dev, torch.float32).contiguous()
        return returns, weight

    def _critic_step(self, k: int, obs: torch.Tensor, act: torch.Tensor, returns: torch.Tensor, weight: torch.Tensor | None,
                     optim: Any, out_loss: torch.Tensor) -> torch.Tensor:
        """``_minimize_critic_squared_loss`` (ddpg.py:267-285): forward, weighted MSE, backward, Adam."""
        B = obs.shape[0]
        st = stream_ptr(self._dev)
        acts, q = self._q_forward(k, obs, act, "cu")
        td = self._buf(f"td{k}", B)
        dq = self._buf("dq", (B, 1))
        rows = self._buf("loss_rows", B)
        call("ts_critic_mse", ptr(q), ptr(returns), ptr(weight), B, ptr(td), ptr(dq), ptr(rows), st)
        call("ts_mean", ptr(rows), B, ptr(out_loss), st)
        self._c[k].backward(acts, dq, B, "cu")
        self._adam(self._g_c[k], optim._optim, optim._max_grad_norm)
        return td

    def _deterministic_actor_step(self, obs: torch.Tensor, out_loss: torch.Tensor) -> None:
        """actor loss -critic(s, actor(s)).mean() (ddpg.py:406, td3.py:216) with the critic's parameters after this update's
        critic step; the critic contributes its input gradient only, so the gradient reaches the actor alone."""
        B, A = obs.shape[0], self.act_dim
        st = stream_ptr(self._dev)
        a_acts = self._actor.forward(obs, B, "au")
        z = a_acts[-1]
        act = self._buf("au_act", (B, A))
        call("ts_det_actor_head", ptr(z), A, B, A, self._max_action, None, 0.0, 0.0, ptr(act), st)
        c_acts, q = self._q_forward(0, obs, act, "aq0")
        dq, rows = self._buf("dq1", (B, 1)), self._buf("loss_rows", B)
        call("ts_det_actor_q_grad", ptr(q), B, ptr(dq), ptr(rows), st)
        call("ts_mean", ptr(rows), B, ptr(out_loss), st)
        dact = self._c[0].backward(c_acts, dq, B, "aq0", param_grads=False, input_grad=True,
                                   input_cols=(self.obs_dim, self.obs_dim + A))
        dz = self._buf("dhead", (B, A))
        call("ts_det_actor_head_bwd", ptr(z), A, ptr(dact), B, A, self._max_action, ptr(dz), st)
        self._actor.backward(a_acts, dz, B, "au")
        self._adam(self._g_actor, self.policy_optim._optim, self.policy_optim._max_grad_norm)

    def _update_lagged_network_weights(self) -> None:
        for tgt, src in self._lagged:
            polyak_update(tgt, src, self.tau)

    # ------------------------------------------------------------------ CUDA-graph mode
    _in_graph_body = False
    _cols_override: Any = None          # the mirror's columns while the graphed body runs (no cross-stream wait inside a capture)

    def _graph_usable(self, buffer: ReplayBuffer) -> bool:
        cols = buffer.device_columns() if hasattr(buffer, "device_columns") else None
        # (a learning-rate schedule would change a constant baked into the captured launches every update: eager then)
        return (self.cuda_graph and not hasattr(buffer, "update_weight") and cols is not None and not self.lr_schedulers
                and buffer._save_obs_next and all(k in cols for k in ("obs", "act", "rew", "terminated", "done", "obs_next")))

    def _graph_variant(self) -> Hashable:
        """Which control flow the next update takes; each variant gets a graph of its own."""
        return None

    def _stats_from_losses(self, losses: np.ndarray) -> TrainingStats:
        """The update's stats from its loss scalars on the host; runs once per update (advances host-side counters)."""
        raise NotImplementedError

    def _device_body(self, buffer: ReplayBuffer, g: dict[str, Any]) -> None:
        """Everything of one update() after the index / noise draws, with no host synchronisation: n-step chain, target,
        critic steps, the actor step, Polyak.  Runs eagerly once, then inside the capture, then as graph replays."""
        from ... import ops
        idx, meta, cols = g["idx"], g["meta"], g["cols"]
        noise_iter = iter(g["noise"])
        saved_fn, self._noise_fn = self._noise_fn, lambda shape: next(noise_iter)
        saved_adam, self._adam = self._adam, FlatGroup.adam_step_device
        self._in_graph_body, self._cols_override = True, cols
        try:
            B = idx.numel()
            n = self.n_step_return_horizon
            stacked = ops.stack_next_indices(meta, idx, n)
            last = stacked[-1].contiguous()
            tq = self._target_q(buffer, last).reshape(B, -1).clone()
            ops.value_mask_rows(tq, cols["terminated"].view(torch.uint8), last)
            rew = cols["rew"] if cols["rew"].dtype == torch.float64 else cols["rew"].to(torch.float64)
            returns = ops.nstep_return(rew, ops.buffer_end_flags(meta), tq, stacked, self.gamma, n, out_dtype=torch.float64)
            batch = Batch()
            batch.__dict__["obs"] = self._rows(buffer, "obs", idx).contiguous()
            batch.__dict__["act"] = self._rows(buffer, "act", idx).contiguous()
            batch.__dict__["returns"] = returns.to(torch.float32)
            self._update_with_batch(batch)
            g["h_losses"].copy_(self._buf("losses", self._n_losses), non_blocking=True)
        finally:
            self._noise_fn, self._adam, self._in_graph_body, self._cols_override = saved_fn, saved_adam, False, None

    def update(self, buffer: ReplayBuffer, sample_size: int | None) -> TrainingStats:
        """``OffPolicyAlgorithm.update`` (algorithm_base.py:868-903); with ``cuda_graph=True`` the device work is one graph replay."""
        if buffer is None or not self.policy.is_within_training_step or not self._graph_usable(buffer):
            return super().update(buffer, sample_size)
        from ...ops import DeviceBufferMeta
        from ...utils.torch_utils import torch_train_mode
        start = time.time()
        dev = self._dev
        indices = np.asarray(buffer.sample_indices(sample_size), dtype=np.int64)
        B, A = len(indices), self.act_dim
        cols = buffer.device_columns()                       # also orders this stream after the mirror's pending copies
        E = int(buffer.buffer_num)
        g = self._graph = self._graphs.setdefault(self._graph_variant(), {})
        key = (B, E, tuple(int(cols[k].data_ptr()) for k in sorted(cols)),
               *(float(o._optim.param_groups[0]["lr"]) for o in self._optimizers))
        if g.get("key") != key:                              # (re)build the persistent inputs; the next call captures
            g.clear()
            g.update(key=key, calls=0, graph=None, cols=dict(cols),
                     h_idx=torch.empty(B, dtype=torch.int64, pin_memory=True), idx=torch.empty(B, dtype=torch.int64, device=dev),
                     h_meta=torch.empty((3, E), dtype=torch.int64, pin_memory=True), d_meta=torch.empty((3, E), dtype=torch.int64, device=dev),
                     noise=torch.empty((self._n_noise, B, A), dtype=torch.float32, device=dev),
                     h_losses=torch.empty(self._n_losses, dtype=torch.float32, pin_memory=True))
            off = torch.from_numpy(np.asarray(buffer._extend_offset, dtype=np.int64)).to(dev)
            g["meta"] = DeviceBufferMeta(off, cols["done"].view(torch.uint8), g["d_meta"][0], g["d_meta"][1], g["d_meta"][2])
        g["h_idx"].numpy()[...] = indices
        hm = g["h_meta"].numpy()
        hm[0], hm[1], hm[2] = buffer.last_index, buffer._sizes, buffer._ins
        g["idx"].copy_(g["h_idx"], non_blocking=True)
        g["d_meta"].copy_(g["h_meta"], non_blocking=True)
        for i in range(self._n_noise):                       # the update's noise draws, in the reference's order
            g["noise"][i].copy_(self._noise_fn((B, A)).to(dev, torch.float32))
        with torch_train_mode(self):
            if g["graph"] is not None:
                g["graph"].replay()
            elif g["calls"] == 0:                            # first update with these shapes: eager (allocates every scratch buffer)
                self._device_body(buffer, g)
            else:                                            # second: capture, then replay it as this update
                graph = torch.cuda.CUDAGraph()
                torch.cuda.synchronize(dev)
                with torch.cuda.graph(graph):
                    self._device_body(buffer, g)
                g["graph"] = graph
                graph.replay()
        g["calls"] += 1
        torch.cuda.current_stream(dev).synchronize()         # the one host sync: the loss scalars
        for sched in self.lr_schedulers:
            sched.step()
        stat = self._stats_from_losses(g["h_losses"].numpy())
        stat.train_time = time.time() - start
        return stat


class DDPG(ActorCriticOffPolicyAlgorithm):
    """Deep Deterministic Policy Gradient (arXiv:1509.02971), reference API (ddpg.py:342-410)."""

    def __init__(self, *, policy: ContinuousDeterministicPolicy, policy_optim: OptimizerFactory, critic: nn.Module,
                 critic_optim: OptimizerFactory, tau: float = 0.005, gamma: float = 0.99, n_step_return_horizon: int = 1,
                 cuda_graph: bool = False) -> None:
        super().__init__(policy=policy, policy_optim=policy_optim, critic=critic, critic_optim=critic_optim, tau=tau, gamma=gamma,
                         n_step_return_horizon=n_step_return_horizon, cuda_graph=cuda_graph)
        self._add_lagged_actor()

    def _update_with_batch(self, batch: Batch) -> DDPGTrainingStats | None:
        obs, act = batch.obs, batch.act
        returns, weight = self._returns_and_weight(batch)
        losses = self._buf("losses", 2)                 # (critic, actor)
        batch.weight = self._critic_step(0, obs, act, returns, weight, self.critic_optim, losses[0:1])     # prio-buffer
        self._deterministic_actor_step(obs, losses[1:2])
        self._update_lagged_network_weights()
        if self._in_graph_body:
            return None                                 # the losses stay on the device; update() reads them after the replay
        return self._stats_from_losses(losses.cpu().numpy())  # the only host sync of the update

    def _stats_from_losses(self, losses: np.ndarray) -> DDPGTrainingStats:
        return DDPGTrainingStats(actor_loss=float(losses[1]), critic_loss=float(losses[0]))
