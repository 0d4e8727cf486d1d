"""TEST INFRASTRUCTURE -- golden vectors for DDPG and TD3 from the UNMODIFIED reference (thu-ml/tianshou 2.0.1 imported
through oracle/ref_shim.py), on the buffer and networks of the SAC goldens (oracle/gen_golden_offpolicy.py).

    python -m oracle.gen_golden_td3_ddpg [td3] [ddpg]     # writes tests/golden/td3_ref*.npz, tests/golden/ddpg_ref*.npz

Captured per ``update()`` (seeds ``torch.manual_seed(100 + u)``, ``np.random.seed(500 + u)`` before update u): sampled
indices, n-step returns, loss scalars, for prioritized replay the IS weights, the TD values passed to ``update_weight`` and
the whole sum tree, and every parameter of every online and lagged network after the step; plus a few ``GaussianNoise``
draws under a fixed numpy seed.  tests/test_td3_ddpg_gpu.py rebuilds identical buffers / weights / seeds with tianshou_b200
and compares the CUDA path; oracle/oracle_det.py is pinned to the same files by tests/test_oracle_td3_ddpg.py.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

from oracle.gen_golden_offpolicy import OUT, named, sac_rollout  # noqa: E402  (imports the reference through the shim)
from gymnasium.spaces import Box  # noqa: E402  (shim stand-in)
from tianshou.algorithm import DDPG, TD3  # noqa: E402
from tianshou.algorithm.modelfree.ddpg import ContinuousDeterministicPolicy  # noqa: E402
from tianshou.algorithm.optim import AdamOptimizerFactory  # noqa: E402
from tianshou.data import Batch, PrioritizedVectorReplayBuffer, VectorReplayBuffer  # noqa: E402
from tianshou.exploration import GaussianNoise  # noqa: E402
from tianshou.utils.net.common import Net  # noqa: E402
from tianshou.utils.net.continuous import ContinuousActorDeterministic, ContinuousCritic  # noqa: E402
from tianshou.utils.torch_utils import policy_within_training_step  # noqa: E402

DET_BASE = dict(obs=23, act=5, hidden=(48, 40), E=4, cap=60, steps=45, bs=64, lr=1e-3, tau=0.005, gamma=0.99, max_action=1.0,
                action_scaling=True, prio=False, alpha=0.6, beta=0.4)
DET_VARIANTS = {
    "td3_ref": dict(DET_BASE, algo="td3", n_step=3, updates=6, update_actor_freq=2, policy_noise=0.2, noise_clip=0.5),
    "td3_ref_b": dict(DET_BASE, algo="td3", n_step=1, updates=4, update_actor_freq=3, policy_noise=0.4, noise_clip=0.0,
                      max_action=2.0, action_scaling=False, prio=True),
    "ddpg_ref": dict(DET_BASE, algo="ddpg", n_step=3, updates=3),
    "ddpg_ref_b": dict(DET_BASE, algo="ddpg", n_step=1, updates=3, prio=True),
}


def build_ref_det(cfg, seed=0):
    torch.manual_seed(seed)
    O, A, H = cfg["obs"], cfg["act"], cfg["hidden"]
    actor = ContinuousActorDeterministic(preprocess_net=Net(state_shape=(O,), hidden_sizes=H), action_shape=(A,),
                                         max_action=cfg["max_action"])
    critics = [ContinuousCritic(preprocess_net=Net(state_shape=(O,), action_shape=(A,), hidden_sizes=H, concat=True))
               for _ in range(2 if cfg["algo"] == "td3" else 1)]
    policy = ContinuousDeterministicPolicy(actor=actor, action_space=Box(-1.0, 1.0, (A,)), exploration_noise="default",
                                           action_scaling=cfg["action_scaling"],
                                           action_bound_method="clip" if cfg["action_scaling"] else None)
    opt = lambda: AdamOptimizerFactory(lr=cfg["lr"])  # noqa: E731
    if cfg["algo"] == "td3":
        algo = TD3(policy=policy, policy_optim=opt(), critic=critics[0], critic_optim=opt(), critic2=critics[1], critic2_optim=opt(),
                   tau=cfg["tau"], gamma=cfg["gamma"], policy_noise=cfg["policy_noise"], update_actor_freq=cfg["update_actor_freq"],
                   noise_clip=cfg["noise_clip"], n_step_return_horizon=cfg["n_step"])
    else:
        algo = DDPG(policy=policy, policy_optim=opt(), critic=critics[0], critic_optim=opt(), tau=cfg["tau"], gamma=cfg["gamma"],
                    n_step_return_horizon=cfg["n_step"])
    return algo, actor, critics


def gen_det(which: str):
    """td3_ref*.npz / ddpg_ref*.npz: per update the sampled indices, n-step returns, losses, (prioritized) IS weights, TD values
    and tree leaves, and every parameter of every online and lagged network after the update."""
    for tag, cfg in DET_VARIANTS.items():
        if cfg["algo"] != which:
            continue
        algo, actor, critics = build_ref_det(cfg)
        out = {"cfg_" + k: np.asarray(v) for k, v in cfg.items() if k != "algo"}
        out.update(named(actor, "p0_actor_"))
        for k, c in enumerate(critics):
            out.update(named(c, f"p0_c{k + 1}_"))
        E = cfg["E"]
        if cfg["prio"]:
            buf = PrioritizedVectorReplayBuffer(E * cfg["cap"], E, alpha=cfg["alpha"], beta=cfg["beta"])
        else:
            buf = VectorReplayBuffer(E * cfg["cap"], E)
        for s in sac_rollout(np.random.default_rng(3), E, cfg["steps"], cfg["obs"], cfg["act"]):
            buf.add(Batch(**s), buffer_ids=np.arange(E))
        for k in ("obs", "act", "rew", "terminated", "truncated", "obs_next", "done"):
            out["buf_" + k] = np.asarray(buf._meta[k]).copy()
        out["meta_last_index"] = np.asarray(buf.last_index, dtype=np.int64)
        out["meta_lengths"] = np.asarray(buf._lengths, dtype=np.int64)
        if cfg["prio"]:
            out["tree_leaves0"] = np.asarray(buf.weight[np.arange(buf.maxsize)]).copy()     # every slot, filled or not
        captured = {}
        orig_pre, orig_post = algo._preprocess_batch, algo._postprocess_batch

        def pre(batch, buffer, indices):
            if cfg["prio"]:
                captured["is_weight"] = np.asarray(batch.weight).copy()
            b = orig_pre(batch, buffer, indices)
            captured["indices"] = np.asarray(indices).copy()
            captured["returns"] = b.returns.detach().numpy().copy()
            return b

        def post(batch, buffer, indices):
            captured["td"] = batch.weight.detach().numpy().copy()
            return orig_post(batch, buffer, indices)

        algo._preprocess_batch, algo._postprocess_batch = pre, post
        nets = {"actor_": actor, "actorold_": algo.actor_old}
        for k, c in enumerate(critics):
            nets[f"c{k + 1}_"] = c
        nets["c1old_"] = algo.critic_old
        if len(critics) == 2:
            nets["c2old_"] = algo.critic2_old
        for u in range(cfg["updates"]):
            torch.manual_seed(100 + u)
            np.random.seed(500 + u)
            with policy_within_training_step(algo.policy):
                stats = algo.update(buffer=buf, sample_size=cfg["bs"])
            o = f"u{u}_"
            out[o + "indices"], out[o + "returns"] = captured["indices"], captured["returns"]
            if which == "td3":
                out[o + "losses"] = np.array([stats.actor_loss, stats.critic1_loss, stats.critic2_loss], dtype=np.float64)
            else:
                out[o + "losses"] = np.array([stats.actor_loss, stats.critic_loss], dtype=np.float64)
            if cfg["prio"]:
                out[o + "is_weight"], out[o + "td"] = captured["is_weight"], captured["td"]
                out[o + "tree_leaves"] = np.asarray(buf.weight[np.arange(buf.maxsize)]).copy()
            for prefix, mod in nets.items():
                # the lagged networks are wrapped (EvalModeModuleWrapper): parameters() of the wrapped module, same order
                out.update(named(mod, o + prefix))
        # exploration noise: the policy's "default" GaussianNoise(sigma=0.1) and an explicit one, numpy's global generator
        np.random.seed(7)
        out["noise_default"] = algo.policy.exploration_noise((3, cfg["act"]))
        out["noise_mu_sigma"] = GaussianNoise(mu=0.25, sigma=0.5)((2, 4))
        np.savez_compressed(os.path.join(OUT, f"{tag}.npz"), **out)
        print(f"{tag}.npz", len(out), "arrays,", os.path.getsize(os.path.join(OUT, f"{tag}.npz")), "bytes; losses u0", out["u0_losses"])


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    for w in sys.argv[1:] or ["td3", "ddpg"]:
        gen_det(w)
