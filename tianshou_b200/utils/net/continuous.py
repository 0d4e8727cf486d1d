"""Deterministic and Gaussian actors, critic heads (API of tianshou/utils/net/continuous.py:32-238)."""
from __future__ import annotations

import warnings
from collections.abc import Sequence
from typing import Any

import numpy as np
import torch
from torch import nn

from ..torch_utils import torch_device
from .common import MLP, ModuleWithVectorOutput, TLinearLayer

SIGMA_MIN = -20
SIGMA_MAX = 2


class ContinuousCritic(ModuleWithVectorOutput):
    """V(s) (or Q(s,a) when ``act`` is given): preprocess net -> ``last`` MLP -> 1."""

    def __init__(self, *, preprocess_net: ModuleWithVectorOutput, hidden_sizes: Sequence[int] = (),
                 linear_layer: TLinearLayer = nn.Linear, flatten_input: bool = True,
                 apply_preprocess_net_to_obs_only: bool = False) -> None:
        super().__init__(output_dim=1)
        self.preprocess = preprocess_net
        self.apply_preprocess_net_to_obs_only = apply_preprocess_net_to_obs_only
        self.last = MLP(input_dim=preprocess_net.get_output_dim(), output_dim=1, hidden_sizes=hidden_sizes,
                        linear_layer=linear_layer, flatten_input=flatten_input)

    def forward(self, obs: np.ndarray | torch.Tensor, act: np.ndarray | torch.Tensor | None = None,
                info: dict[str, Any] | None = None) -> torch.Tensor:
        device = torch_device(self)
        obs = torch.as_tensor(obs, device=device, dtype=torch.float32)
        if self.apply_preprocess_net_to_obs_only:
            obs, _ = self.preprocess(obs)
        obs = obs.flatten(1)
        if act is not None:
            act = torch.as_tensor(act, device=device, dtype=torch.float32).flatten(1)
            obs = torch.cat([obs, act], dim=1)
        if not self.apply_preprocess_net_to_obs_only:
            obs, _ = self.preprocess(obs)
        return self.last(obs)


class ContinuousActorDeterministic(ModuleWithVectorOutput):
    """Actions directly (DDPG / TD3): preprocess net -> ``last`` MLP -> ``max_action * tanh`` (continuous.py:32-85)."""

    def __init__(self, *, preprocess_net: ModuleWithVectorOutput, action_shape: Any, hidden_sizes: Sequence[int] = (),
                 max_action: float = 1.0) -> None:
        super().__init__(int(np.prod(action_shape)))
        self.preprocess = preprocess_net
        self.last = MLP(input_dim=preprocess_net.get_output_dim(), output_dim=self.output_dim, hidden_sizes=hidden_sizes)
        self.max_action = max_action

    def get_preprocess_net(self) -> ModuleWithVectorOutput:
        return self.preprocess

    def forward(self, obs: Any, state: Any = None, info: dict[str, Any] | None = None) -> tuple[torch.Tensor, Any]:
        action, hidden = self.preprocess(obs, state)
        return self.max_action * torch.tanh(self.last(action)), hidden


class ContinuousActorProbabilistic(ModuleWithVectorOutput):
    """(mu, sigma) of a diagonal Gaussian; sigma is ``exp(sigma_param)`` (state independent) unless
    ``conditioned_sigma``."""

    def __init__(self, *, preprocess_net: ModuleWithVectorOutput, action_shape: Any,
                 hidden_sizes: Sequence[int] = (), max_action: float = 1.0, unbounded: bool = False,
                 conditioned_sigma: bool = False) -> None:
        output_dim = int(np.prod(action_shape))
        super().__init__(output_dim)
        if unbounded and not np.isclose(max_action, 1.0):
            warnings.warn("Note that max_action input will be discarded when unbounded is True.")
            max_action = 1.0
        self.preprocess = preprocess_net
        input_dim = preprocess_net.get_output_dim()
        self.mu = MLP(input_dim=input_dim, output_dim=output_dim, hidden_sizes=hidden_sizes)
        self._c_sigma = conditioned_sigma
        if conditioned_sigma:
            self.sigma = MLP(input_dim=input_dim, output_dim=output_dim, hidden_sizes=hidden_sizes)
        else:
            self.sigma_param = nn.Parameter(torch.zeros(output_dim, 1))
        self.max_action = max_action
        self._unbounded = unbounded

    def get_preprocess_net(self) -> ModuleWithVectorOutput:
        return self.preprocess

    def forward(self, obs: Any, state: Any = None, info: dict[str, Any] | None = None
                ) -> tuple[tuple[torch.Tensor, torch.Tensor], Any]:
        logits, _hidden = self.preprocess(obs, state)
        mu = self.mu(logits)
        if not self._unbounded:
            mu = self.max_action * torch.tanh(mu)
        if self._c_sigma:
            sigma = torch.clamp(self.sigma(logits), min=SIGMA_MIN, max=SIGMA_MAX).exp()
        else:
            shape = [1] * len(mu.shape)
            shape[1] = -1
            sigma = (self.sigma_param.view(shape) + torch.zeros_like(mu)).exp()
        return (mu, sigma), state
