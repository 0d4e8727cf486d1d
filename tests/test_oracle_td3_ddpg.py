"""Pin the torch-CPU restatement of DDPG / TD3 (oracle/oracle_det.py) to outputs of the imported reference
(tests/golden/td3_ref*.npz, ddpg_ref*.npz), check GaussianNoise against the reference's draws, and check that the fused
algorithms refuse networks that are not on a CUDA device.  CPU only."""
import numpy as np
import pytest
import torch

from oracle import oracle_det as od
from ts_testutil import Box, load_golden

VARIANTS = ["td3_ref", "td3_ref_b", "ddpg_ref", "ddpg_ref_b"]


def _load(params, g, prefix):
    with torch.no_grad():
        for i, p in enumerate(params):
            p.copy_(torch.as_tensor(g[f"{prefix}{i}"]).reshape(p.shape))


def _close(params, g, prefix, lr, what):
    for i, p in enumerate(params):
        np.testing.assert_allclose(p.detach().numpy(), g[f"{prefix}{i}"], rtol=1e-3, atol=0.1 * lr, err_msg=f"{what} {prefix}{i}")


def _host_buffer(g):
    E, cap = int(g["cfg_E"]), int(g["cfg_cap"])
    return dict(obs=g["buf_obs"], act=g["buf_act"], rew=g["buf_rew"], done=g["buf_done"], terminated=g["buf_terminated"],
                obs_next=g["buf_obs_next"], offset=np.arange(E + 1) * cap, last_index=g["meta_last_index"], lengths=g["meta_lengths"])


@pytest.mark.parametrize("name", VARIANTS)
def test_det_oracle_matches_reference_run(name):
    g = load_golden(f"{name}.npz")
    td3 = name.startswith("td3")
    O, A, H = int(g["cfg_obs"]), int(g["cfg_act"]), tuple(int(x) for x in g["cfg_hidden"])
    lr, B, prio = float(g["cfg_lr"]), int(g["cfg_bs"]), bool(g["cfg_prio"])
    n_c = 2 if td3 else 1
    nets = od.DetNets(O, A, H, n_c, max_action=float(g["cfg_max_action"]))
    _load(nets.actor.parameters(), g, "p0_actor_")
    for k in range(n_c):
        _load(nets.c[k].parameters(), g, f"p0_c{k + 1}_")
    nets.sync_lagged()
    opts = [torch.optim.Adam(nets.actor.parameters(), lr=lr)] + [torch.optim.Adam(c.parameters(), lr=lr) for c in nets.c]
    buf = _host_buffer(g)
    gamma, n_step, tau = float(g["cfg_gamma"]), int(g["cfg_n_step"]), float(g["cfg_tau"])
    last_actor_loss = 0.0
    for u in range(int(g["cfg_updates"])):
        o = f"u{u}_"
        w = g[o + "is_weight"] if prio else None
        if td3:
            torch.manual_seed(100 + u)
            noise = torch.randn(B, A)               # td3.py:196: the one torch draw of the update
            due = u % int(g["cfg_update_actor_freq"]) == 0
            res = od.td3_update(nets, opts, buf, g[o + "indices"], noise, float(g["cfg_policy_noise"]), float(g["cfg_noise_clip"]),
                                gamma, n_step, tau, due, is_weight=w)
            if due:
                last_actor_loss = res["actor_loss"]
            got = [last_actor_loss, *res["critic_losses"]]
        else:
            res = od.ddpg_update(nets, opts, buf, g[o + "indices"], gamma, n_step, tau, is_weight=w)
            got = [res["actor_loss"], *res["critic_losses"]]
        np.testing.assert_allclose(res["returns"], g[o + "returns"].reshape(-1), rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(got, g[o + "losses"], rtol=1e-5, atol=1e-6)
        if prio:
            np.testing.assert_allclose(res["td"], g[o + "td"], rtol=1e-4, atol=1e-5)
        _close(nets.actor.parameters(), g, o + "actor_", lr, "actor")
        _close(nets.actor_old.parameters(), g, o + "actorold_", lr, "lagged actor")
        for k in range(n_c):
            _close(nets.c[k].parameters(), g, o + f"c{k + 1}_", lr, "critic")
            _close(nets.c_old[k].parameters(), g, o + f"c{k + 1}old_", lr, "lagged critic")


def test_td3_golden_lagged_networks_move_only_with_the_actor():
    """td3_ref.npz (update_actor_freq 2): the lagged networks are Polyak-updated on updates 0, 2, 4 only."""
    g = load_golden("td3_ref.npz")
    for u in range(1, int(g["cfg_updates"])):
        for net in ("actorold_", "c1old_", "c2old_"):
            same = all(np.array_equal(g[f"u{u}_{net}{i}"], g[f"u{u - 1}_{net}{i}"]) for i in range(4))
            assert same == (u % 2 == 1), (u, net)


@pytest.mark.parametrize("name", VARIANTS)
def test_gaussian_noise_matches_reference_draws(name):
    from tianshou_b200.exploration import BaseNoise, GaussianNoise
    g = load_golden(f"{name}.npz")
    np.random.seed(7)
    noise = GaussianNoise(sigma=0.1)
    assert isinstance(noise, BaseNoise)
    np.testing.assert_array_equal(noise((3, int(g["cfg_act"]))), g["noise_default"])
    np.testing.assert_array_equal(GaussianNoise(mu=0.25, sigma=0.5)((2, 4)), g["noise_mu_sigma"])
    noise.reset()
    with pytest.raises(AssertionError):
        GaussianNoise(sigma=-1.0)


@pytest.mark.parametrize("algo_name", ["td3", "ddpg"])
def test_cpu_networks_are_refused(algo_name):
    from tianshou_b200.algorithm import AdamOptimizerFactory, UnsupportedModelError
    from tianshou_b200.algorithm.modelfree.ddpg import DDPG, ContinuousDeterministicPolicy
    from tianshou_b200.algorithm.modelfree.td3 import TD3
    from tianshou_b200.utils.net.common import Net
    from tianshou_b200.utils.net.continuous import ContinuousActorDeterministic, ContinuousCritic
    actor = ContinuousActorDeterministic(preprocess_net=Net(state_shape=(6,), hidden_sizes=(16,)), action_shape=(2,))
    critic = ContinuousCritic(preprocess_net=Net(state_shape=(6,), action_shape=(2,), hidden_sizes=(16,), concat=True))
    policy = ContinuousDeterministicPolicy(actor=actor, action_space=Box(2), exploration_noise="default")
    cls = TD3 if algo_name == "td3" else DDPG
    with pytest.raises(UnsupportedModelError, match="no CPU path"):
        cls(policy=policy, policy_optim=AdamOptimizerFactory(lr=1e-3), critic=critic, critic_optim=AdamOptimizerFactory(lr=1e-3))


def test_deterministic_policy_cpu_forward_and_noise():
    """The Collector's path of ContinuousDeterministicPolicy is plain torch: usable without a GPU."""
    from tianshou_b200.algorithm.modelfree.ddpg import ContinuousDeterministicPolicy
    from tianshou_b200.data import Batch
    from tianshou_b200.exploration import GaussianNoise
    from tianshou_b200.utils.net.common import Net
    from tianshou_b200.utils.net.continuous import ContinuousActorDeterministic
    torch.manual_seed(0)
    actor = ContinuousActorDeterministic(preprocess_net=Net(state_shape=(6,), hidden_sizes=(16,)), action_shape=(3,), max_action=2.0)
    with pytest.warns(UserWarning, match="max_action=2.0"):
        policy = ContinuousDeterministicPolicy(actor=actor, action_space=Box(3), exploration_noise="default")
    assert isinstance(policy.exploration_noise, GaussianNoise) and policy.exploration_noise._sigma == 0.1
    out = policy(Batch(obs=np.random.default_rng(0).standard_normal((5, 6)).astype(np.float32), info=Batch()))
    assert out.act.shape == (5, 3) and float(out.act.abs().max()) <= 2.0
