"""TEST INFRASTRUCTURE -- torch restatement (plain torch, autograd) of the reference's DDPG and TD3 update bodies.

Only ``tests/`` and ``tools/td3_ddpg_bench.py`` may import this module; ``tianshou_b200`` never does.  Like
``oracle/oracle_offpolicy.py`` (whose n-step helpers it reuses) it restates the reference without the framework around it,
each step citing the reference lines (paths relative to the reference's ``tianshou/`` package):

  DDPG : algorithm/modelfree/ddpg.py:266-285 (critic squared loss), :314-339 (target value), :396-410 (update)
  TD3  : algorithm/modelfree/td3.py:94-102 (min of the lagged critics), :190-226 (smoothing, delayed actor, update)
  both : utils/net/continuous.py:70-85 (deterministic actor), utils/lagged_network.py:8-18 (Polyak)

Every function takes the networks on a ``device``: the CPU for the restatement pinned to the goldens, a GPU for the
eager-PyTorch context number of ``tools/td3_ddpg_bench.py``.

PINNING: tests/test_oracle_td3_ddpg.py replays tests/golden/td3_ref*.npz / ddpg_ref*.npz (outputs of the imported reference,
oracle/gen_golden_td3_ddpg.py) through these functions: returns, losses, TD values and post-update parameters must match.
"""
from __future__ import annotations

import copy

import numpy as np
import torch
from torch import nn

from .oracle_offpolicy import compute_nstep_targets, mlp


class DetNets:
    """ContinuousActorDeterministic + 1 (DDPG) or 2 (TD3) ContinuousCritics with lagged copies of all of them, in the reference
    modules' ``parameters()`` order: actor = preprocess, last; critic = preprocess, last.  ``device``: where the torch code runs
    (CPU for the pinned restatement, a GPU for the eager-PyTorch context number of tools/td3_ddpg_bench.py)."""

    def __init__(self, obs: int, act: int, hidden: tuple[int, ...], n_critics: int, max_action: float = 1.0, device: str = "cpu"):
        self.device = torch.device(device)
        self.max_action = max_action
        self.actor = nn.Sequential(mlp([obs, *hidden], True), nn.Linear(hidden[-1], act)).to(self.device)
        self.c = [nn.Sequential(mlp([obs + act, *hidden], True), nn.Linear(hidden[-1], 1)).to(self.device) for _ in range(n_critics)]
        self.sync_lagged()

    def sync_lagged(self) -> None:
        self.actor_old = copy.deepcopy(self.actor)
        self.c_old = [copy.deepcopy(c) for c in self.c]

    def act(self, obs: torch.Tensor, old: bool = False) -> torch.Tensor:
        """ContinuousActorDeterministic.forward (utils/net/continuous.py:70-85)."""
        return self.max_action * torch.tanh((self.actor_old if old else self.actor)(obs))


def _critic_step(critic: nn.Module, opt: torch.optim.Optimizer, obs: torch.Tensor, act: torch.Tensor, returns: torch.Tensor,
                 weight: torch.Tensor | float) -> tuple[float, torch.Tensor]:
    """``_minimize_critic_squared_loss`` (ddpg.py:266-285)."""
    td = critic(torch.cat([obs, act], dim=1)).flatten() - returns
    loss = (td.pow(2) * weight).mean()
    opt.zero_grad(); loss.backward(); opt.step()
    return loss.item(), td.detach()


def _actor_step(nets: DetNets, opt: torch.optim.Optimizer, obs: torch.Tensor) -> float:
    """-critic(obs, actor(obs)).mean() with critic 1 (ddpg.py:406, td3.py:216); only the actor's optimiser steps."""
    loss = -nets.c[0](torch.cat([obs, nets.act(obs)], dim=1)).mean()
    opt.zero_grad(); loss.backward(); opt.step()
    return loss.item()


def _polyak(nets: DetNets, tau: float) -> None:
    """``_update_lagged_network_weights`` (utils/lagged_network.py:8-18) on every lagged network."""
    with torch.no_grad():
        for tgt, src in [(nets.actor_old, nets.actor), *zip(nets.c_old, nets.c)]:
            for t, s in zip(tgt.parameters(), src.parameters(), strict=True):
                t.copy_(tau * s + (1 - tau) * t)


def _det_update(nets: DetNets, opts: list[torch.optim.Optimizer], buf: dict, indices: np.ndarray, is_weight: np.ndarray | None,
                noise: torch.Tensor | None, policy_noise: float, noise_clip: float, gamma: float, n_step: int, tau: float,
                actor_step: bool) -> dict:
    dev = nets.device

    def target_q(terminal: np.ndarray) -> torch.Tensor:
        obs_next = torch.from_numpy(buf["obs_next"][terminal]).to(dev)
        a = nets.act(obs_next, old=True)                              # lagged actor (ddpg.py:400-402)
        if noise is not None:                                         # target-policy smoothing (td3.py:190-202)
            n = noise.to(dev) * policy_noise
            if noise_clip > 0.0:
                n = n.clamp(-noise_clip, noise_clip)
            a = a + n
        x = torch.cat([obs_next, a], dim=1)
        return torch.stack([c(x) for c in nets.c_old]).min(dim=0)[0].cpu()      # td3.py:94-102 (one critic: itself)

    returns = torch.from_numpy(compute_nstep_targets(buf, indices, target_q, gamma, n_step)).flatten().to(dev)
    obs, act = torch.from_numpy(buf["obs"][indices]).to(dev), torch.from_numpy(buf["act"][indices]).to(dev)
    weight = torch.as_tensor(is_weight, dtype=torch.float32, device=dev) if is_weight is not None else 1.0
    losses, tds = [], []
    for k, c in enumerate(nets.c):
        loss, td = _critic_step(c, opts[1 + k], obs, act, returns, weight)
        losses.append(loss); tds.append(td)
    actor_loss = None
    if actor_step:
        actor_loss = _actor_step(nets, opts[0], obs)
        _polyak(nets, tau)
    return dict(returns=returns.cpu().numpy(), critic_losses=losses, actor_loss=actor_loss,
                td=(sum(tds) / len(tds)).cpu().numpy())


def ddpg_update(nets: DetNets, opts: list[torch.optim.Optimizer], buf: dict, indices: np.ndarray, gamma: float, n_step: int,
                tau: float, is_weight: np.ndarray | None = None) -> dict:
    """One ``DDPG.update`` on ``indices`` (ddpg.py:396-410): target critic_old(s', actor_old(s')), critic step, actor step,
    Polyak on critic_old and actor_old.  ``opts`` = [actor, critic]; ``td`` is what the prioritized buffer receives."""
    return _det_update(nets, opts, buf, indices, is_weight, None, 0.0, 0.0, gamma, n_step, tau, True)


def td3_update(nets: DetNets, opts: list[torch.optim.Optimizer], buf: dict, indices: np.ndarray, noise: torch.Tensor,
               policy_noise: float, noise_clip: float, gamma: float, n_step: int, tau: float, actor_step: bool,
               is_weight: np.ndarray | None = None) -> dict:
    """One ``TD3.update`` on ``indices`` (td3.py:190-226) with the (B, A) standard-normal smoothing draw given: both critic
    steps; when ``actor_step`` (``_cnt % update_actor_freq == 0``) the actor step and Polyak on all three lagged networks.
    ``opts`` = [actor, critic1, critic2]; ``td`` = (td1 + td2) / 2."""
    return _det_update(nets, opts, buf, indices, is_weight, noise, policy_noise, noise_clip, gamma, n_step, tau, actor_step)
