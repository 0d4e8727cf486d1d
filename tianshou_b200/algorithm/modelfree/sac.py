"""Soft Actor-Critic with the whole ``update()`` on the device (SURVEY 8(f) rank 2, BASELINE configs[3]).

Reference: tianshou/algorithm/modelfree/sac.py (SACPolicy :55-131, Alpha :133-215, SAC :218-336),
modelfree/td3.py:31-102 (dual critics, ``min`` target), modelfree/ddpg.py:196-339 (n-step target, critic
squared loss), utils/lagged_network.py:8-80 (Polyak).

Per ``update(buffer, sample_size)``:
  host : index draw (``buffer.sample_indices``: numpy RandomState streams, SURVEY A9 -- kept so the sampled
         transitions are the reference's), the two ``rsample`` noise draws (torch generator), one D2H of 3 loss scalars.
  GPU  : row gathers from the buffer's device mirror (or one upload of the sampled rows), target actor + lagged critics
         forward -> ``ts_sac_target`` -> ``ts_nstep_return``; per critic forward / loss / backward (``ts_net_gemm``) + Adam;
         actor forward, critics' input-gradient GEMMs, tanh-Gaussian head backward, actor backward + Adam; Polyak axpy.
Every Linear layer's forward / input gradient / weight gradient is one tcgen05 GEMM launch (csrc/net_gemm.cu).
The row gathers, critic step, Polyak update and CUDA-graph mode are shared with DDPG / TD3 (ddpg.py, td3.py).
"""
from __future__ import annotations

from abc import ABC, abstractmethod
from dataclasses import dataclass
from typing import Any, Union

import numpy as np
import torch
from torch import nn
from torch.distributions import Independent, Normal

from ..._cabi import call, ptr, stream_ptr
from ...data import Batch, ReplayBuffer
from ..base import Policy, TrainingStats
from ..flat_params import UnsupportedModelError
from ..netgraph import ACT_NONE, _Layer
from ..optim import OptimizerFactory
from .ddpg import _linear_relu_chain, describe_q_critic  # noqa: F401  (describe_q_critic: re-exported)
from .td3 import ActorDualCriticsOffPolicyAlgorithm

SIGMA_MIN, SIGMA_MAX = -20.0, 2.0          # utils/net/continuous.py:17-18
_F32_EPS = float(np.finfo(np.float32).eps)


def correct_log_prob_gaussian_tanh(log_prob: torch.Tensor, tanh_squashed_action: torch.Tensor,
                                   eps: float = _F32_EPS) -> torch.Tensor:
    """Equation 21 of arXiv:1801.01290 (sac.py:25-39)."""
    return log_prob - torch.log(1 - tanh_squashed_action.pow(2) + eps).sum(-1, keepdim=True)


@dataclass(kw_only=True)
class SACTrainingStats(TrainingStats):
    actor_loss: float
    critic1_loss: float
    critic2_loss: float
    alpha: float | None = None
    alpha_loss: float | None = None


class SACPolicy(Policy):
    """Tanh-squashed Gaussian policy (sac.py:55-131).  ``forward`` is the torch-module path the Collector runs."""

    def __init__(self, *, actor: nn.Module, exploration_noise: Any = None, deterministic_eval: bool = True,
                 action_scaling: bool = True, action_space: Any, observation_space: Any | None = None) -> None:
        super().__init__(action_space=action_space, observation_space=observation_space, action_scaling=action_scaling,
                         action_bound_method=None)
        if exploration_noise == "default":
            raise UnsupportedModelError("exploration_noise='default' (GaussianNoise) is not provided; pass a callable or None")
        self.actor = actor
        self.exploration_noise = exploration_noise
        self.deterministic_eval = deterministic_eval

    def add_exploration_noise(self, act: Any, batch: Any) -> Any:
        if self.exploration_noise is None:
            return act
        if isinstance(act, np.ndarray):
            return act + self.exploration_noise(act.shape)
        return act

    def forward(self, batch: Batch, state: Any = None, **kwargs: Any) -> Batch:
        (loc, scale), hidden = self.actor(batch.obs, state=state, info=batch.get("info"))
        dist = Independent(Normal(loc=loc, scale=scale), 1)
        act = dist.mode if (self.deterministic_eval and not self.is_within_training_step) else dist.rsample()
        log_prob = dist.log_prob(act).unsqueeze(-1)
        squashed = torch.tanh(act)
        log_prob = correct_log_prob_gaussian_tanh(log_prob, squashed)
        return Batch(logits=(loc, scale), act=squashed, state=hidden, dist=dist, log_prob=log_prob)


class Alpha(ABC):
    """Entropy regularisation coefficient (sac.py:133-165)."""

    @staticmethod
    def from_float_or_instance(alpha: Union[float, "Alpha"]) -> "Alpha":
        if isinstance(alpha, float):
            return FixedAlpha(alpha)
        if isinstance(alpha, Alpha):
            return alpha
        raise ValueError(f"Expected float or Alpha instance, but got {alpha=}")

    @property
    @abstractmethod
    def value(self) -> float: ...

    @abstractmethod
    def update(self, entropy: torch.Tensor) -> float | None: ...


class FixedAlpha(Alpha):
    def __init__(self, alpha: float):
        self._value = alpha

    @property
    def value(self) -> float:
        return self._value

    def update(self, entropy: torch.Tensor) -> float | None:
        return None


class AutoAlpha(nn.Module, Alpha):
    """Auto-tuned alpha (sac.py:168-215): a single scalar parameter; its three-flop update stays in torch."""

    def __init__(self, target_entropy: float, log_alpha: float, optim: OptimizerFactory):
        super().__init__()
        self._target_entropy = target_entropy
        self._log_alpha = nn.Parameter(torch.tensor(log_alpha))
        self._optim, lr_scheduler = optim.create_instances(self)
        if lr_scheduler is not None:
            raise ValueError(f"Learning rate schedulers are not supported by {self.__class__.__name__}")

    @property
    def value(self) -> float:
        return self._log_alpha.detach().exp().item()

    def update(self, entropy: torch.Tensor) -> float:
        entropy_deficit = self._target_entropy - entropy.to(self._log_alpha.device)
        alpha_loss = -(self._log_alpha * entropy_deficit).mean()
        self._optim.zero_grad()
        alpha_loss.backward()
        self._optim.step()
        return alpha_loss.item()


# ------------------------------------------------------------------------------------------------ module -> kernel views
def describe_gaussian_actor(actor: Any, obs_dim: int) -> tuple[list[_Layer], list[nn.Parameter], int]:
    """ContinuousActorProbabilistic(conditioned_sigma=True, unbounded=True): trunk + ONE virtual head layer whose rows are
    (mu.weight ; sigma.weight) -- adjacent in the flat buffer, so the head is a single [2A, H] GEMM."""
    if not getattr(actor, "_c_sigma", False):
        raise UnsupportedModelError("SAC actor: conditioned_sigma=True expected (examples/mujoco/mujoco_sac.py:97-104)")
    if not getattr(actor, "_unbounded", False):
        raise UnsupportedModelError("SAC actor: only unbounded=True (mu without tanh) is supported")
    trunk = _linear_relu_chain(actor.preprocess, obs_dim, "actor.preprocess")
    mu = _linear_relu_chain(actor.mu, trunk[-1].out_dim, "actor.mu")
    sg = _linear_relu_chain(actor.sigma, trunk[-1].out_dim, "actor.sigma")
    if len(mu) != 1 or len(sg) != 1 or mu[0].out_dim != sg[0].out_dim:
        raise UnsupportedModelError("SAC actor: mu / sigma heads must be single Linear layers of equal width")
    A = mu[0].out_dim
    params: list[nn.Parameter] = []
    for L in trunk:
        params += [L.weight, L.bias]
    params += [mu[0].weight, sg[0].weight, mu[0].bias, sg[0].bias]     # adjacency = the virtual [2A, H] layer
    head = _Layer("linear", mu[0].weight, mu[0].bias, ACT_NONE, mu[0].in_dim, 2 * A)
    return [*trunk, head], params, A


class SAC(ActorDualCriticsOffPolicyAlgorithm):
    """Soft Actor-Critic (arXiv:1801.01290 / 1812.05905), reference API (sac.py:218-336)."""

    _n_noise = 2        # the two rsample draws: target action, then the actor step's action
    _n_losses = 3

    def __init__(self, *, policy: SACPolicy, policy_optim: OptimizerFactory, critic: nn.Module, critic_optim: OptimizerFactory,
                 critic2: nn.Module | None = None, critic2_optim: OptimizerFactory | None = None, tau: float = 0.005,
                 gamma: float = 0.99, alpha: float | Alpha = 0.2, n_step_return_horizon: int = 1,
                 deterministic_eval: bool = True, cuda_graph: bool = False) -> None:
        super().__init__(policy=policy, policy_optim=policy_optim, critic=critic, critic_optim=critic_optim, critic2=critic2,
                         critic2_optim=critic2_optim, tau=tau, gamma=gamma, n_step_return_horizon=n_step_return_horizon,
                         cuda_graph=cuda_graph)
        self.deterministic_eval = deterministic_eval
        self.alpha = Alpha.from_float_or_instance(alpha)

    def _describe_actor(self, actor: nn.Module) -> tuple[list[_Layer], list[nn.Parameter], int]:
        return describe_gaussian_actor(actor, self.obs_dim)

    # ------------------------------------------------------------------ helpers
    def _actor_forward(self, obs: torch.Tensor, tag: str) -> tuple[list[torch.Tensor], torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
        """policy(batch) on the device: returns (activations, act, log_prob, sigma, noise)."""
        B, A = obs.shape[0], self.act_dim
        acts = self._actor.forward(obs, B, tag)
        head = acts[-1]
        noise = self._noise_fn((B, A)).to(self._dev, torch.float32).contiguous()
        act = self._buf(tag + "_act", (B, A))
        logp = self._buf(tag + "_logp", B)
        sigma = self._buf(tag + "_sigma", (B, A))
        call("ts_squashed_gaussian", ptr(head), 2 * A, ptr(noise), B, A, SIGMA_MIN, SIGMA_MAX, _F32_EPS, ptr(act), ptr(logp),
             ptr(sigma), stream_ptr(self._dev))
        return acts, act, logp, sigma, noise

    # ------------------------------------------------------------------ target
    def _target_q(self, buffer: ReplayBuffer, indices: np.ndarray) -> torch.Tensor:
        """min(Q1', Q2')(s', a') - alpha * log pi(a'|s') with a' ~ pi(.|s')   (ddpg.py:327-339, td3.py:94-102, sac.py:298-302)"""
        obs_next = self._obs_next(buffer, indices)
        B = obs_next.shape[0]
        _, act, logp, _, _ = self._actor_forward(obs_next, "tq")
        _, q1 = self._q_forward(0, obs_next, act, "tq", target=True)
        _, q2 = self._q_forward(1, obs_next, act, "tq", target=True)
        out = self._buf("tq_out", (B, 1))
        call("ts_sac_target", ptr(q1), ptr(q2), ptr(logp), float(self.alpha.value), B, ptr(out), stream_ptr(self._dev))
        return out

    # ------------------------------------------------------------------ update
    def _update_with_batch(self, batch: Batch) -> SACTrainingStats | None:
        st = stream_ptr(self._dev)
        obs, act = batch.obs, batch.act
        B, A = obs.shape[0], self.act_dim
        returns, weight = self._returns_and_weight(batch)
        losses = self._buf("losses", 3)
        td1 = self._critic_step(0, obs, act, returns, weight, self.critic_optim, losses[0:1])
        td2 = self._critic_step(1, obs, act, returns, weight, self.critic2_optim, losses[1:2])
        batch.weight = (td1 + td2) / 2.0       # prio-buffer

        # actor: L = mean(alpha * log pi(a|s) - min(Q1, Q2)(s, a)),  a = tanh(mu + sigma * eps)
        alpha = float(self.alpha.value)
        a_acts, new_act, logp, sigma, noise = self._actor_forward(obs, "au")
        c1_acts, q1a = self._q_forward(0, obs, new_act, "aq0")
        c2_acts, q2a = self._q_forward(1, obs, new_act, "aq1")
        dq1, dq2, rows = self._buf("dq1", (B, 1)), self._buf("dq2", (B, 1)), self._buf("loss_rows", B)
        call("ts_sac_actor_q_grad", ptr(q1a), ptr(q2a), ptr(logp), alpha, B, ptr(dq1), ptr(dq2), ptr(rows), st)
        call("ts_mean", ptr(rows), B, ptr(losses[2:3]), st)
        cols = (self.obs_dim, self.obs_dim + A)
        da1 = self._c[0].backward(c1_acts, dq1, B, "aq0", param_grads=False, input_grad=True, input_cols=cols)
        da2 = self._c[1].backward(c2_acts, dq2, B, "aq1", param_grads=False, input_grad=True, input_cols=cols)
        dact = da1 + da2
        dhead = self._buf("dhead", (B, 2 * A))
        call("ts_squashed_gaussian_bwd", ptr(a_acts[-1]), 2 * A, ptr(noise), ptr(new_act), ptr(sigma), ptr(dact), B, A,
             SIGMA_MIN, SIGMA_MAX, _F32_EPS, alpha / B, ptr(dhead), st)
        self._actor.backward(a_acts, dhead, B, "au")
        self._adam(self._g_actor, self.policy_optim._optim, self.policy_optim._max_grad_norm)

        alpha_loss = None if self._in_graph_body else self.alpha.update(-logp.detach().unsqueeze(-1))
        self._update_lagged_network_weights()
        if self._in_graph_body:
            return None                         # the losses stay on the device; update() reads them after the replay
        return self._stats_from_losses(losses.cpu().numpy(), alpha_loss)      # the only host sync of the update

    def _stats_from_losses(self, losses: np.ndarray, alpha_loss: float | None = None) -> SACTrainingStats:
        return SACTrainingStats(actor_loss=float(losses[2]), critic1_loss=float(losses[0]), critic2_loss=float(losses[1]),
                                alpha=float(self.alpha.value), alpha_loss=alpha_loss)

    # ------------------------------------------------------------------ CUDA-graph mode
    def _graph_usable(self, buffer: ReplayBuffer) -> bool:
        return isinstance(self.alpha, FixedAlpha) and super()._graph_usable(buffer)
