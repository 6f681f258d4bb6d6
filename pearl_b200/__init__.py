"""pearl_b200 — B200-native (sm_100a) learner hot path of facebookresearch/Pearl:
`ReplayBuffer.sample -> PolicyLearner.learn()` behind Pearl's own plugin API.

    from pearl_b200 import B200ReplayBuffer, B200DeepQLearning, B200DoubleDQN

Hand-written CUDA in libpearlb200.so (C ABI: include/pearl_b200.h), called through
ctypes; PyTorch only allocates memory and provides streams.  No CPU fallback.
"""
from ._compat import HAVE_PEARL, OneHotActionTensorRepresentationModule, TransitionBatch  # noqa: F401
from .dqn import B200DeepQLearning, B200DoubleDQN, B200LearnerGroup  # noqa: F401
from .replay_buffer import B200ReplayBuffer  # noqa: F401
from .per import B200PrioritizedReplayBuffer  # noqa: F401
from .her import B200HindsightExperienceReplayBuffer  # noqa: F401
from .ppo import gae_and_lambda_returns  # noqa: F401
# subclasses of the reference's ContinuousSoftActorCritic / SoftActorCritic / ProximalPolicyOptimization / TD3 / DDPG when Pearl
# is importable,
# the stand-alone CUDA learners (same keyword arguments) otherwise
from .actor_critic import (B200ContinuousSoftActorCritic, B200DeepDeterministicPolicyGradient,  # noqa: F401
                           B200ProximalPolicyOptimization, B200SoftActorCritic, B200TD3)
from .dist import B200Communicator, all_gather_bytes, shard_owner  # noqa: F401

__all__ = ["B200ReplayBuffer", "B200DeepQLearning", "B200DoubleDQN", "TransitionBatch",
           "OneHotActionTensorRepresentationModule", "HAVE_PEARL", "B200Communicator", "B200LearnerGroup", "B200PrioritizedReplayBuffer", "gae_and_lambda_returns", "B200ContinuousSoftActorCritic", "B200SoftActorCritic", "B200ProximalPolicyOptimization",
           "B200TD3", "B200DeepDeterministicPolicyGradient", "B200HindsightExperienceReplayBuffer"]
