"""TD3 with the whole ``update()`` on the device, and the dual-critic base that TD3 and SAC share.

Reference: tianshou/algorithm/modelfree/td3.py (ActorDualCriticsOffPolicyAlgorithm :31-102, TD3 :105-226).

Per ``update(buffer, sample_size)``:
  host : index draw (``buffer.sample_indices``), one (B, A) standard-normal draw for target-policy smoothing (torch generator
         of the networks' device), one D2H of the loss scalars.
  GPU  : lagged actor forward -> ``ts_det_actor_head`` (smoothing noise) -> both lagged critics -> ``ts_sac_target`` (min,
         no entropy term) -> ``ts_nstep_return``; both critic steps; every ``update_actor_freq``-th update the actor step
         (critic 1 only) and Polyak on all three lagged networks.
"""
from __future__ import annotations

from collections.abc import Hashable
from copy import deepcopy
from dataclasses import dataclass

import numpy as np
import torch
from torch import nn

from ..._cabi import call, ptr, stream_ptr
from ...data import Batch
from ..base import Policy, TrainingStats
from ..optim import OptimizerFactory
from .ddpg import ActorCriticOffPolicyAlgorithm, ContinuousDeterministicPolicy


@dataclass(kw_only=True)
class TD3TrainingStats(TrainingStats):
    actor_loss: float
    critic1_loss: float
    critic2_loss: float


class ActorDualCriticsOffPolicyAlgorithm(ActorCriticOffPolicyAlgorithm):
    """Two critics with lagged copies; the target value is the minimum of the lagged critics (td3.py:31-102)."""

    def __init__(self, *, policy: Policy, policy_optim: OptimizerFactory, critic: nn.Module, critic_optim: OptimizerFactory,
                 critic2: nn.Module | None = None, critic2_optim: OptimizerFactory | None = None, tau: float = 0.005,
                 gamma: float = 0.99, n_step_return_horizon: int = 1, cuda_graph: bool = False) -> None:
        super().__init__(policy=policy, policy_optim=policy_optim, critic=critic, critic_optim=critic_optim, tau=tau, gamma=gamma,
                         n_step_return_horizon=n_step_return_horizon, cuda_graph=cuda_graph)
        self.critic2 = critic2 or deepcopy(critic)
        self.critic2_old = self._add_critic(self.critic2)
        self.critic2_optim = self._fused_optimizer(self.critic2, critic2_optim or critic_optim, self._g_c[1])

    def _target_q_compute_value(self, obs_next: torch.Tensor, act: torch.Tensor) -> torch.Tensor:
        """min(Q1', Q2')(s', a')   (td3.py:94-102)"""
        B = obs_next.shape[0]
        _, q1 = self._q_forward(0, obs_next, act, "tq", target=True)
        _, q2 = self._q_forward(1, obs_next, act, "tq", target=True)
        out = self._buf("tq_out", (B, 1))
        call("ts_sac_target", ptr(q1), ptr(q2), None, 0.0, B, ptr(out), stream_ptr(self._dev))
        return out


class TD3(ActorDualCriticsOffPolicyAlgorithm):
    """Twin Delayed DDPG (arXiv:1802.09477), reference API (td3.py:105-226)."""

    _n_noise = 1
    _n_losses = 3

    def __init__(self, *, policy: ContinuousDeterministicPolicy, policy_optim: OptimizerFactory, critic: nn.Module,
                 critic_optim: OptimizerFactory, critic2: nn.Module | None = None, critic2_optim: OptimizerFactory | None = None,
                 tau: float = 0.005, gamma: float = 0.99, policy_noise: float = 0.2, update_actor_freq: int = 2,
                 noise_clip: float = 0.5, n_step_return_horizon: int = 1, cuda_graph: bool = False) -> None:
        super().__init__(policy=policy, policy_optim=policy_optim, critic=critic, critic_optim=critic_optim, critic2=critic2,
                         critic2_optim=critic2_optim, tau=tau, gamma=gamma, n_step_return_horizon=n_step_return_horizon,
                         cuda_graph=cuda_graph)
        self._add_lagged_actor()
        self.policy_noise = policy_noise
        self.update_actor_freq = update_actor_freq
        self.noise_clip = noise_clip
        self._cnt = 0
        self._last = 0.0

    def _target_smoothing(self, B: int) -> tuple[torch.Tensor | None, float, float]:
        noise = self._noise_fn((B, self.act_dim)).to(self._dev, torch.float32).contiguous()
        return noise, float(self.policy_noise), float(self.noise_clip)

    def _actor_due(self) -> bool:
        return self._cnt % self.update_actor_freq == 0

    def _graph_variant(self) -> Hashable:
        return self._actor_due()          # critic-only updates and critic + actor + Polyak updates are two graphs

    def _update_with_batch(self, batch: Batch) -> TD3TrainingStats | None:
        obs, act = batch.obs, batch.act
        returns, weight = self._returns_and_weight(batch)
        losses = self._buf("losses", 3)                 # (critic1, critic2, actor)
        td1 = self._critic_step(0, obs, act, returns, weight, self.critic_optim, losses[0:1])
        td2 = self._critic_step(1, obs, act, returns, weight, self.critic2_optim, losses[1:2])
        batch.weight = (td1 + td2) / 2.0                # prio-buffer
        if self._actor_due():                           # delayed actor update, then all three lagged networks (td3.py:215-219)
            self._deterministic_actor_step(obs, losses[2:3])
            self._update_lagged_network_weights()
        if self._in_graph_body:
            return None                                 # the losses stay on the device; update() reads them after the replay
        return self._stats_from_losses(losses.cpu().numpy())     # the only host sync of the update

    def _stats_from_losses(self, losses: np.ndarray) -> TD3TrainingStats:
        if self._actor_due():
            self._last = float(losses[2])
        self._cnt += 1
        return TD3TrainingStats(actor_loss=self._last, critic1_loss=float(losses[0]), critic2_loss=float(losses[1]))
