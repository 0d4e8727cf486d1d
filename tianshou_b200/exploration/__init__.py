"""Action noise for exploration (API of tianshou/exploration/random.py:7-32)."""
from .random import BaseNoise, GaussianNoise

__all__ = ["BaseNoise", "GaussianNoise"]
