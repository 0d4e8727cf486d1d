"""TEST INFRASTRUCTURE -- golden vectors for the off-policy update bodies (SURVEY 8(f) ranks 2-3) from the UNMODIFIED
reference (thu-ml/tianshou 2.0.1 imported from /root/reference through oracle/ref_shim.py).

    python -m oracle.gen_golden_offpolicy          # writes tests/golden/sac_ref.npz, tests/golden/dqn_ref*.npz

Captured per ``update()``: sampled indices, n-step returns, loss scalars, TD errors, every parameter tensor of every
network (online and lagged) after the step.  The tests rebuild identical buffers / weights / seeds with tianshou_b200 and
compare the CUDA path; ``oracle/oracle_offpolicy.py`` (torch-CPU restatement, the CPU arm of the bench) is pinned to
the same files.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden")

from oracle.ref_shim import import_reference  # noqa: E402

ts = import_reference()
from gymnasium.spaces import Box, Discrete  # noqa: E402  (shim stand-ins)
from tianshou.algorithm import DQN, SAC  # noqa: E402
from tianshou.algorithm.modelfree.dqn import DiscreteQLearningPolicy  # noqa: E402
from tianshou.algorithm.modelfree.sac import SACPolicy  # noqa: E402
from tianshou.algorithm.optim import AdamOptimizerFactory  # noqa: E402
from tianshou.data import Batch, PrioritizedVectorReplayBuffer, VectorReplayBuffer  # noqa: E402
from tianshou.env.atari.atari_network import DQNet, ScaledObsInputActionReprNet  # noqa: E402
from tianshou.utils.net.common import Net  # noqa: E402
from tianshou.utils.net.continuous import ContinuousActorProbabilistic, ContinuousCritic  # noqa: E402
from tianshou.utils.torch_utils import policy_within_training_step  # noqa: E402


def named(mod: torch.nn.Module, prefix: str) -> dict[str, np.ndarray]:
    return {f"{prefix}{i}": p.detach().numpy().copy() for i, p in enumerate(mod.parameters())}


# ---------------------------------------------------------------------------------------------------------- SAC
SAC_CFG = dict(obs=23, act=5, hidden=(48, 40), E=4, cap=60, steps=45, bs=64, n_step=3, updates=3, lr=1e-3, tau=0.005,
               gamma=0.99, alpha=0.2)


def sac_rollout(rng, E, steps, obs_dim, act_dim):
    out = []
    obs = rng.standard_normal((E, obs_dim)).astype(np.float32)
    for _ in range(steps):
        act = np.tanh(rng.standard_normal((E, act_dim))).astype(np.float32)
        rew = rng.standard_normal(E)
        obs_next = rng.standard_normal((E, obs_dim)).astype(np.float32)
        term = rng.random(E) < 0.06
        trunc = (rng.random(E) < 0.04) & ~term
        out.append(dict(obs=obs, act=act, rew=rew, terminated=term, truncated=trunc, obs_next=obs_next))
        done = term | trunc
        obs = np.where(done[:, None], rng.standard_normal((E, obs_dim)).astype(np.float32), obs_next)
    return out


def build_ref_sac(cfg, seed=0):
    torch.manual_seed(seed)
    O, A, H = cfg["obs"], cfg["act"], cfg["hidden"]
    net_a = Net(state_shape=(O,), hidden_sizes=H)
    actor = ContinuousActorProbabilistic(preprocess_net=net_a, action_shape=(A,), unbounded=True, conditioned_sigma=True)
    c1 = ContinuousCritic(preprocess_net=Net(state_shape=(O,), action_shape=(A,), hidden_sizes=H, concat=True))
    c2 = ContinuousCritic(preprocess_net=Net(state_shape=(O,), action_shape=(A,), hidden_sizes=H, concat=True))
    policy = SACPolicy(actor=actor, action_space=Box(-1.0, 1.0, (A,)))
    algo = SAC(policy=policy, policy_optim=AdamOptimizerFactory(lr=cfg["lr"]), critic=c1, critic_optim=AdamOptimizerFactory(lr=cfg["lr"]),
               critic2=c2, critic2_optim=AdamOptimizerFactory(lr=cfg["lr"]), tau=cfg["tau"], gamma=cfg["gamma"], alpha=cfg["alpha"],
               n_step_return_horizon=cfg["n_step"])
    return algo, actor, c1, c2


def gen_sac():
    cfg = SAC_CFG
    algo, actor, c1, c2 = build_ref_sac(cfg)
    out = {"cfg_" + k: np.asarray(v) for k, v in cfg.items()}
    out.update(named(actor, "p0_actor_")); out.update(named(c1, "p0_c1_")); out.update(named(c2, "p0_c2_"))
    buf = VectorReplayBuffer(cfg["E"] * cfg["cap"], cfg["E"])
    roll = sac_rollout(np.random.default_rng(3), cfg["E"], cfg["steps"], cfg["obs"], cfg["act"])
    for s in roll:
        buf.add(Batch(**s), buffer_ids=np.arange(cfg["E"]))
    for k in ("obs", "act", "rew", "terminated", "truncated", "obs_next", "done"):
        out["buf_" + k] = np.asarray(buf._meta[k]).copy()
    out["meta_last_index"] = np.asarray(buf.last_index, dtype=np.int64)
    out["meta_lengths"] = np.asarray(buf._lengths, dtype=np.int64)
    captured = {}
    orig_pre = algo._preprocess_batch

    def pre(batch, buffer, indices):
        b = orig_pre(batch, buffer, indices)
        captured["indices"] = np.asarray(indices).copy()
        captured["returns"] = b.returns.detach().numpy().copy()
        return b

    algo._preprocess_batch = pre
    for u in range(cfg["updates"]):
        torch.manual_seed(100 + u)
        with policy_within_training_step(algo.policy):
            stats = algo.update(buffer=buf, sample_size=cfg["bs"])
        o = f"u{u}_"
        out[o + "indices"], out[o + "returns"] = captured["indices"], captured["returns"]
        out[o + "losses"] = np.array([stats.actor_loss, stats.critic1_loss, stats.critic2_loss], dtype=np.float64)
        out.update(named(actor, o + "actor_")); out.update(named(c1, o + "c1_")); out.update(named(c2, o + "c2_"))
        out.update(named(algo.critic_old, o + "c1old_")); out.update(named(algo.critic2_old, o + "c2old_"))
    np.savez_compressed(os.path.join(OUT, "sac_ref.npz"), **out)
    print("sac_ref.npz", len(out), "arrays; losses u0", out["u0_losses"])


# ---------------------------------------------------------------------------------------------------------- DQN
DQN_VARIANTS = {
    "": dict(H=36, W=36, A=5, E=4, cap=64, steps=50, bs=16, n_step=3, updates=5, lr=1e-3, gamma=0.99, target_freq=2, is_double=True,
             huber=None, alpha=0.6, beta=0.4),
    "_b": dict(H=36, W=36, A=3, E=2, cap=48, steps=40, bs=8, n_step=1, updates=3, lr=5e-4, gamma=0.9, target_freq=3, is_double=False,
               huber=1.0, alpha=0.5, beta=0.4),
}


def dqn_rollout(rng, E, steps, H, W, A):
    out = []
    frame = rng.integers(0, 256, (E, H, W), dtype=np.uint8)
    stack = np.repeat(frame[:, None], 4, axis=1)
    for _ in range(steps):
        act = rng.integers(0, A, E)
        rew = rng.standard_normal(E)
        term = rng.random(E) < 0.08
        trunc = (rng.random(E) < 0.03) & ~term
        nxt = rng.integers(0, 256, (E, H, W), dtype=np.uint8)
        stack_next = np.concatenate([stack[:, 1:], nxt[:, None]], axis=1)
        out.append(dict(obs=stack.copy(), act=act, rew=rew, terminated=term, truncated=trunc, obs_next=stack_next.copy()))
        done = term | trunc
        fresh = rng.integers(0, 256, (E, H, W), dtype=np.uint8)
        stack = np.where(done[:, None, None, None], np.repeat(fresh[:, None], 4, axis=1), stack_next)
    return out


def build_ref_dqn(cfg, seed=0):
    torch.manual_seed(seed)
    net = ScaledObsInputActionReprNet(DQNet(4, cfg["H"], cfg["W"], cfg["A"]))
    policy = DiscreteQLearningPolicy(model=net, action_space=Discrete(cfg["A"]))
    algo = DQN(policy=policy, optim=AdamOptimizerFactory(lr=cfg["lr"]), gamma=cfg["gamma"], n_step_return_horizon=cfg["n_step"],
               target_update_freq=cfg["target_freq"], is_double=cfg["is_double"], huber_loss_delta=cfg["huber"])
    return algo, net


def gen_dqn():
    for tag, cfg in DQN_VARIANTS.items():
        algo, net = build_ref_dqn(cfg)
        out = {"cfg_" + k: np.asarray(np.nan if v is None else v) for k, v in cfg.items()}
        out.update(named(net, "p0_q_"))
        buf = PrioritizedVectorReplayBuffer(cfg["E"] * cfg["cap"], cfg["E"], alpha=cfg["alpha"], beta=cfg["beta"], stack_num=4,
                                            ignore_obs_next=True, save_only_last_obs=True)
        roll = dqn_rollout(np.random.default_rng(8), cfg["E"], cfg["steps"], cfg["H"], cfg["W"], cfg["A"])
        for i, s in enumerate(roll):
            for k in ("obs", "act", "rew", "terminated", "truncated", "obs_next"):
                if k != "obs_next":     # ignore_obs_next: never stored; the replay passes a dummy
                    out[f"roll{i}_{k}"] = s[k] if k != "obs" else s[k][:, -1]     # last frame only (what is stored)
            buf.add(Batch(**s), buffer_ids=np.arange(cfg["E"]))
        out["roll_first_stack"] = roll[0]["obs"]
        captured = {}
        orig_pre, orig_post = algo._preprocess_batch, algo._postprocess_batch

        def pre(batch, buffer, indices):
            b = orig_pre(batch, buffer, indices)
            captured["indices"] = np.asarray(indices).copy()
            captured["returns"] = b.returns.detach().numpy().copy()
            captured["is_weight"] = np.asarray(batch.weight).copy()
            return b

        def post(batch, buffer, indices):
            captured["td"] = batch.weight.detach().numpy().copy()
            return orig_post(batch, buffer, indices)

        algo._preprocess_batch, algo._postprocess_batch = pre, post
        for u in range(cfg["updates"]):
            np.random.seed(500 + u)
            with policy_within_training_step(algo.policy):
                stats = algo.update(buffer=buf, sample_size=cfg["bs"])
            o = f"u{u}_"
            out[o + "indices"], out[o + "returns"], out[o + "td"] = captured["indices"], captured["returns"], captured["td"]
            out[o + "is_weight"] = captured["is_weight"]
            out[o + "loss"] = np.float64(stats.loss)
            if u == cfg["updates"] - 1:      # parameters after the LAST update only (every earlier step feeds into them)
                out.update(named(net, o + "q_"))
                if algo.model_old is not None:
                    out.update(named(algo.model_old, o + "qold_"))
            out[o + "tree_root"] = np.float64(buf.weight.reduce())
            out[o + "tree_leaves"] = np.asarray(buf.weight[np.arange(len(buf))]).copy()
        params = {k: out.pop(k) for k in [k for k in out if k.startswith(f"u{cfg['updates'] - 1}_q")]}
        np.savez_compressed(os.path.join(OUT, f"dqn_ref{tag}.npz"), **out)
        np.savez_compressed(os.path.join(OUT, f"dqn_ref{tag}_params.npz"), **params)     # apart: every file stays under 1 MB
        print(f"dqn_ref{tag}.npz", len(out), "arrays; losses", [float(out[f'u{u}_loss']) for u in range(cfg['updates'])])


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    which = sys.argv[1:] or ["sac", "dqn"]
    for w in which:
        {"sac": gen_sac, "dqn": gen_dqn}[w]()
