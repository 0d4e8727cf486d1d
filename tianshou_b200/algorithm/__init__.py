from .base import Algorithm, OffPolicyAlgorithm, OnPolicyAlgorithm, Policy, TrainingStats
from .flat_params import UnsupportedModelError
from .modelfree.a2c import A2CTrainingStats, ActorCriticOnPolicyAlgorithm
from .modelfree.ddpg import DDPG
from .modelfree.ppo import A2C, PPO
from .modelfree.reinforce import DiscreteActorPolicy, ProbabilisticActorPolicy
from .modelfree.td3 import TD3
from .optim import AdamOptimizerFactory, LRSchedulerFactoryLinear, OptimizerFactory, RMSpropOptimizerFactory

__all__ = [
    "Algorithm", "OffPolicyAlgorithm", "OnPolicyAlgorithm", "Policy", "TrainingStats",
    "UnsupportedModelError", "A2CTrainingStats", "ActorCriticOnPolicyAlgorithm", "PPO", "A2C", "DDPG", "TD3",
    "ProbabilisticActorPolicy", "DiscreteActorPolicy", "AdamOptimizerFactory", "LRSchedulerFactoryLinear", "OptimizerFactory",
    "RMSpropOptimizerFactory",
]
