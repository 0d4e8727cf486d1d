"""Exploration noise added to numpy actions by ``add_exploration_noise`` (exploration/random.py:7-32).  Draws come from
numpy's global generator, as in the reference, so a seeded run reproduces the reference's noise."""
from __future__ import annotations

from abc import ABC, abstractmethod
from collections.abc import Sequence

import numpy as np


class BaseNoise(ABC):
    """The action noise base class."""

    @abstractmethod
    def reset(self) -> None:
        """Reset to the initial state."""

    @abstractmethod
    def __call__(self, size: Sequence[int]) -> np.ndarray:
        """Generate new noise."""


class GaussianNoise(BaseNoise):
    """i.i.d. N(mu, sigma^2) per action element; the default exploration noise of DDPG / TD3."""

    def __init__(self, mu: float = 0.0, sigma: float = 1.0) -> None:
        assert sigma >= 0, "Noise std should not be negative."
        self._mu = mu
        self._sigma = sigma

    def __call__(self, size: Sequence[int]) -> np.ndarray:
        return np.random.normal(self._mu, self._sigma, size)

    def reset(self) -> None:
        pass
