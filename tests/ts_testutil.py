"""Shared helpers for the test-suite (golden fixture loading, model construction)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def load_golden(name: str):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def load_dqn_golden(variant: str) -> dict:
    """``dqn_ref{variant}.npz`` together with ``dqn_ref{variant}_params.npz`` (the network parameters after the last
    update, stored in a file of their own so that no fixture file exceeds 1 MB)."""
    return {**load_golden(f"dqn_ref{variant}.npz"), **load_golden(f"dqn_ref{variant}_params.npz")}


PARAM_ORDER = ["a_w1", "a_b1", "a_w2", "a_b2", "a_w3", "a_b3", "a_logstd",
               "c_w1", "c_b1", "c_w2", "c_b2", "c_w3", "c_b3"]


class Box:
    """Minimal stand-in for gymnasium.spaces.Box (gymnasium is not a dependency)."""

    def __init__(self, dim: int):
        self.shape = (dim,)
        self.low = -np.ones(dim, np.float32)
        self.high = np.ones(dim, np.float32)


def build_actor_critic(obs_dim: int, act_dim: int, device, seed: int = 0):
    import torch

    from tianshou_b200.utils.net.common import Net
    from tianshou_b200.utils.net.continuous import ContinuousActorProbabilistic, ContinuousCritic

    torch.manual_seed(seed)
    net_a = Net(state_shape=(obs_dim,), hidden_sizes=(64, 64), activation=torch.nn.Tanh)
    actor = ContinuousActorProbabilistic(preprocess_net=net_a, action_shape=(act_dim,), unbounded=True).to(device)
    net_c = Net(state_shape=(obs_dim,), hidden_sizes=(64, 64), activation=torch.nn.Tanh)
    critic = ContinuousCritic(preprocess_net=net_c).to(device)
    torch.nn.init.constant_(actor.sigma_param, -0.5)
    for m in list(actor.modules()) + list(critic.modules()):
        if isinstance(m, torch.nn.Linear):
            torch.nn.init.orthogonal_(m.weight, gain=np.sqrt(2))
            torch.nn.init.zeros_(m.bias)
    for m in actor.mu.modules():
        if isinstance(m, torch.nn.Linear):
            torch.nn.init.zeros_(m.bias)
            m.weight.data.copy_(0.01 * m.weight.data)
    return actor, critic


def named_params(actor, critic):
    import torch
    a1, a2 = [m for m in actor.preprocess.model.model if isinstance(m, torch.nn.Linear)]
    c1, c2 = [m for m in critic.preprocess.model.model if isinstance(m, torch.nn.Linear)]
    a3, c3 = actor.mu.model[0], critic.last.model[0]
    return {"a_w1": a1.weight, "a_b1": a1.bias, "a_w2": a2.weight, "a_b2": a2.bias, "a_w3": a3.weight,
            "a_b3": a3.bias, "a_logstd": actor.sigma_param, "c_w1": c1.weight, "c_b1": c1.bias, "c_w2": c2.weight,
            "c_b2": c2.bias, "c_w3": c3.weight, "c_b3": c3.bias}


def load_params(actor, critic, values: dict) -> None:
    import torch
    with torch.no_grad():
        for k, p in named_params(actor, critic).items():
            p.copy_(torch.as_tensor(values[k]).reshape(p.shape))


def gaussian_dist(loc_scale):
    import torch
    loc, scale = loc_scale
    return torch.distributions.Independent(torch.distributions.Normal(loc, scale), 1)


def build_ppo(obs_dim, act_dim, device, lr=3e-4, params=None, **kw):
    from tianshou_b200.algorithm import PPO, AdamOptimizerFactory, ProbabilisticActorPolicy
    actor, critic = build_actor_critic(obs_dim, act_dim, device)
    if params is not None:
        load_params(actor, critic, params)
    policy = ProbabilisticActorPolicy(actor=actor, dist_fn=gaussian_dist, action_scaling=True,
                                      action_bound_method="clip", action_space=Box(act_dim))
    algo = PPO(policy=policy, critic=critic, optim=AdamOptimizerFactory(lr=lr), **kw)
    return algo, actor, critic


def restore_vector_buffer(g, prefix: str, E: int, cap: int, device=None):
    """Rebuild a tianshou_b200 VectorReplayBuffer in the exact state stored in a golden file."""
    from tianshou_b200.data import Batch, VectorReplayBuffer
    buf = VectorReplayBuffer(E * cap, E, device=device)
    meta = Batch(obs=g[prefix + "buf_obs"].copy(), act=g[prefix + "buf_act"].copy(), rew=g[prefix + "buf_rew"].copy(),
                 terminated=g[prefix + "buf_terminated"].copy(), truncated=g[prefix + "buf_truncated"].copy(),
                 done=g[prefix + "buf_done"].copy(), obs_next=g[prefix + "buf_obs_next"].copy())
    buf.set_batch(meta)
    set_buffer_state(buf, g[prefix + "meta_last_index"], g[prefix + "meta_lengths"])
    return buf


def set_buffer_state(buf, last_index, lengths) -> None:
    buf.last_index[:] = last_index
    buf._sizes[:] = lengths
    buf._ins[:] = np.where(lengths > 0, (last_index - buf._offset + 1) % buf._cap, 0)
    buf._touch()


def synth_rollout(rng, E, steps, obs_dim, act_dim, p_term=1e-3, trunc_len=1000):
    """Synthetic HalfCheetah-shaped rollout (SURVEY 8d); yields per-step dicts of [E, ...] arrays."""
    t_in_ep = np.zeros(E, dtype=np.int64)
    obs = rng.standard_normal((E, obs_dim)).astype(np.float32)
    for _ in range(steps):
        act = rng.standard_normal((E, act_dim)).astype(np.float32)
        rew = rng.standard_normal(E)
        obs_next = rng.standard_normal((E, obs_dim)).astype(np.float32)
        term = rng.random(E) < p_term
        t_in_ep += 1
        trunc = (t_in_ep >= trunc_len) & ~term
        yield dict(obs=obs, act=act, rew=rew, terminated=term, truncated=trunc, obs_next=obs_next)
        done = term | trunc
        t_in_ep[done] = 0
        obs = np.where(done[:, None], rng.standard_normal((E, obs_dim)).astype(np.float32), obs_next)


# ---- observed-error bookkeeping: every parity test records what it measured; tests/conftest.py dumps the table to
# gpurun_out/parity_report.json at the end of the session (copied to profiles/ per round)
PARITY: dict = {}


def record_parity(key: str, got, ref, rtol: float, atol: float) -> dict:
    """Assert ``|got - ref| <= atol + rtol * |ref|`` elementwise and record the observed errors under ``key``."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape, f"{key}: shape {got.shape} vs {ref.shape}"
    err = np.abs(got - ref)
    scale = float(np.abs(ref).max()) if ref.size else 0.0
    worst = float((err - (atol + rtol * np.abs(ref))).max()) if ref.size else 0.0
    e = {"n": int(ref.size), "max_abs_err": float(err.max()) if ref.size else 0.0, "max_abs_ref": scale,
         "max_err_over_max_ref": float(err.max() / scale) if scale > 0 else 0.0,
         "rtol": rtol, "atol": atol, "margin": -worst, "ok": bool(worst <= 0.0)}
    prev = PARITY.get(key)
    if prev is None or e["max_err_over_max_ref"] >= prev["max_err_over_max_ref"]:
        PARITY[key] = e
    assert worst <= 0.0, (f"{key}: max |err| {e['max_abs_err']:.3e} (max |ref| {scale:.3e}, ratio {e['max_err_over_max_ref']:.3e}) "
                          f"exceeds atol {atol:g} + rtol {rtol:g} * |ref| by {worst:.3e}")
    return e
