"""TD3 / DDPG update bodies on the GPU vs outputs of the imported reference (tests/golden/td3_ref*.npz, ddpg_ref*.npz from
oracle/gen_golden_td3_ddpg.py: same initial weights, same buffer contents, same numpy / torch seeds): sampled indices
bit-exact, n-step returns, losses, (prioritized) IS weights, TD values and tree leaves, and the parameters of every online
and lagged network after each update; eager and CUDA-graph mode, the Collector path and a state_dict round trip."""
import numpy as np
import pytest
import torch

from ts_testutil import Box, load_golden, record_parity, set_buffer_state

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
COLS = ("obs", "act", "rew", "terminated", "truncated", "done", "obs_next")


def _load(mod, g, prefix):
    with torch.no_grad():
        for i, p in enumerate(mod.parameters()):
            p.copy_(torch.as_tensor(g[f"{prefix}{i}"]).reshape(p.shape))


def _check_params(tag, mod, g, prefix, lr):
    for i, p in enumerate(mod.parameters()):
        # Adam normalises the step to ~lr per element: the absolute term is stated in units of one step
        record_parity(f"{tag}/{prefix}{i}", p.detach().cpu().numpy(), g[f"{prefix}{i}"], rtol=1e-3, atol=0.1 * lr)


def _build(g, td3, **kw):
    from tianshou_b200.algorithm import AdamOptimizerFactory
    from tianshou_b200.algorithm.modelfree.ddpg import DDPG, ContinuousDeterministicPolicy
    from tianshou_b200.algorithm.modelfree.td3 import TD3
    from tianshou_b200.utils.net.common import Net
    from tianshou_b200.utils.net.continuous import ContinuousActorDeterministic, ContinuousCritic
    O, A, H = int(g["cfg_obs"]), int(g["cfg_act"]), tuple(int(x) for x in g["cfg_hidden"])
    lr, scaling = float(g["cfg_lr"]), bool(g["cfg_action_scaling"])
    actor = ContinuousActorDeterministic(preprocess_net=Net(state_shape=(O,), hidden_sizes=H), action_shape=(A,),
                                         max_action=float(g["cfg_max_action"])).to(DEV)
    critics = [ContinuousCritic(preprocess_net=Net(state_shape=(O,), action_shape=(A,), hidden_sizes=H, concat=True)).to(DEV)
               for _ in range(2 if td3 else 1)]
    _load(actor, g, "p0_actor_")
    for k, c in enumerate(critics):
        _load(c, g, f"p0_c{k + 1}_")
    policy = ContinuousDeterministicPolicy(actor=actor, action_space=Box(A), exploration_noise="default", action_scaling=scaling,
                                           action_bound_method="clip" if scaling else None)
    common = dict(policy=policy, policy_optim=AdamOptimizerFactory(lr=lr), critic=critics[0], critic_optim=AdamOptimizerFactory(lr=lr),
                  tau=float(g["cfg_tau"]), gamma=float(g["cfg_gamma"]), n_step_return_horizon=int(g["cfg_n_step"]), **kw)
    if td3:
        algo = TD3(critic2=critics[1], critic2_optim=AdamOptimizerFactory(lr=lr), policy_noise=float(g["cfg_policy_noise"]),
                   update_actor_freq=int(g["cfg_update_actor_freq"]), noise_clip=float(g["cfg_noise_clip"]), **common)
    else:
        algo = DDPG(**common)
    # the reference ran on the CPU and drew its smoothing noise from torch's CPU generator: same draws, uploaded
    algo._noise_fn = lambda shape: torch.normal(torch.zeros(shape), torch.ones(shape)).to(DEV)
    return algo, actor, critics, lr


def _buffer(g, mirror):
    from tianshou_b200.data import Batch, PrioritizedVectorReplayBuffer, VectorReplayBuffer
    E, cap = int(g["cfg_E"]), int(g["cfg_cap"])
    if bool(g["cfg_prio"]):
        buf = PrioritizedVectorReplayBuffer(E * cap, E, alpha=float(g["cfg_alpha"]), beta=float(g["cfg_beta"]), device=DEV,
                                            device_mirror=mirror)
    else:
        buf = VectorReplayBuffer(E * cap, E, device=DEV, device_mirror=mirror)
    buf.set_batch(Batch(**{k: g["buf_" + k].copy() for k in COLS}))
    set_buffer_state(buf, g["meta_last_index"], g["meta_lengths"])
    if bool(g["cfg_prio"]):
        buf.weight[np.arange(buf.maxsize)] = g["tree_leaves0"]
    if mirror:
        buf.sync_device_mirror()
        assert buf.device_columns() is not None
    return buf


def _nets(algo, actor, critics):
    out = {"actor_": actor, "actorold_": algo.actor_old, "c1old_": algo.critic_old}
    for k, c in enumerate(critics):
        out[f"c{k + 1}_"] = c
    if len(critics) == 2:
        out["c2old_"] = algo.critic2_old
    return out


def _stat_losses(stats, td3):
    if td3:
        return np.array([stats.actor_loss, stats.critic1_loss, stats.critic2_loss])
    return np.array([stats.actor_loss, stats.critic_loss])


@pytest.mark.parametrize("mirror", [False, True])
@pytest.mark.parametrize("name", ["td3_ref", "td3_ref_b", "ddpg_ref", "ddpg_ref_b"])
def test_update_matches_reference(name, mirror):
    from tianshou_b200.utils import policy_within_training_step
    g = load_golden(f"{name}.npz")
    td3, prio = name.startswith("td3"), bool(g["cfg_prio"])
    algo, actor, critics, lr = _build(g, td3)
    buf = _buffer(g, mirror)
    captured = {}
    orig_pre, orig_post = algo._preprocess_batch, algo._postprocess_batch

    def pre(batch, buffer, indices):
        if prio:
            captured["is_weight"] = batch.weight.detach().cpu().numpy().copy()
        b = orig_pre(batch, buffer, indices)
        captured["indices"], captured["returns"] = np.asarray(indices).copy(), b.returns.detach().cpu().numpy().copy()
        return b

    def post(batch, buffer, indices):
        captured["td"] = batch.weight.detach().cpu().numpy().copy()
        return orig_post(batch, buffer, indices)

    algo._preprocess_batch, algo._postprocess_batch = pre, post
    nets = _nets(algo, actor, critics)
    for u in range(int(g["cfg_updates"])):
        torch.manual_seed(100 + u)
        np.random.seed(500 + u)
        with policy_within_training_step(algo.policy):
            stats = algo.update(buffer=buf, sample_size=int(g["cfg_bs"]))
        o, tag = f"u{u}_", f"{name}_m{int(mirror)}_u{u}"
        assert np.array_equal(captured["indices"], g[o + "indices"]), f"update {u}: sampled indices differ from the reference's"
        ref_ret = g[o + "returns"]
        record_parity(f"{tag}/returns", captured["returns"].reshape(ref_ret.shape), ref_ret, rtol=1e-5,
                      atol=1e-5 * float(np.abs(ref_ret).max()))
        record_parity(f"{tag}/losses", _stat_losses(stats, td3), g[o + "losses"], rtol=2e-5, atol=2e-6)
        if prio:
            record_parity(f"{tag}/is_weight", captured["is_weight"], g[o + "is_weight"], rtol=1e-4, atol=1e-6)
            record_parity(f"{tag}/td", captured["td"], g[o + "td"], rtol=1e-5, atol=2e-5 * float(np.abs(g[o + "td"]).max()))
            # leaves are (|td| + eps) ** alpha: a TD value near zero carries the TD's absolute error through the power
            leaves = g[o + "tree_leaves"]
            record_parity(f"{tag}/tree_leaves", np.asarray(buf.weight[np.arange(buf.maxsize)]), leaves, rtol=1e-4,
                          atol=2e-5 * float(np.abs(leaves).max()))
        for prefix, mod in nets.items():
            _check_params(tag, mod, g, o + prefix, lr)
        assert stats.train_time > 0
    if td3:
        assert algo._cnt == int(g["cfg_updates"])


@pytest.mark.parametrize("name", ["td3_ref", "ddpg_ref"])
def test_cuda_graph_matches_reference(name):
    """``cuda_graph=True``: the first update of each control-flow variant runs eagerly, the second is captured and replayed,
    later ones are replays.  TD3 (update_actor_freq 2) has two graphs: critic only, and critic + actor + Polyak."""
    from tianshou_b200.utils import policy_within_training_step
    g = load_golden(f"{name}.npz")
    td3 = name.startswith("td3")
    algo, actor, critics, lr = _build(g, td3, cuda_graph=True)
    buf = _buffer(g, True)
    nets = _nets(algo, actor, critics)
    n_up = int(g["cfg_updates"])
    for u in range(n_up):
        torch.manual_seed(100 + u)
        np.random.seed(500 + u)
        with policy_within_training_step(algo.policy):
            stats = algo.update(buffer=buf, sample_size=int(g["cfg_bs"]))
        o, tag = f"u{u}_", f"{name}_graph_u{u}"
        assert np.array_equal(algo._graph["h_idx"].numpy(), g[o + "indices"]), "sampled indices differ from the reference's"
        record_parity(f"{tag}/losses", _stat_losses(stats, td3), g[o + "losses"], rtol=2e-5, atol=2e-6)
        for prefix, mod in nets.items():
            _check_params(tag, mod, g, o + prefix, lr)
    if td3:
        assert set(algo._graphs) == {True, False} and all(v["graph"] is not None for v in algo._graphs.values())
        assert algo._cnt == n_up
        actor_steps = (n_up + 1) // 2
    else:
        assert algo._graph["graph"] is not None and algo._graph["calls"] == n_up
        actor_steps = n_up
    for grp in algo._g_c:
        grp.sync_step_from_device()
        assert grp.step == n_up
    algo._g_actor.sync_step_from_device()
    assert algo._g_actor.step == actor_steps


def test_collector_path_bounds_and_exploration_noise():
    """``policy(batch)`` (the Collector's call) on the torch modules, ``map_action`` clipping, ``add_exploration_noise``."""
    from tianshou_b200.data import Batch
    from tianshou_b200.exploration import GaussianNoise
    for name in ("td3_ref", "td3_ref_b"):
        g = load_golden(f"{name}.npz")
        algo, actor, *_ = _build(g, True)
        O, A, max_action = int(g["cfg_obs"]), int(g["cfg_act"]), float(g["cfg_max_action"])
        obs = np.random.default_rng(0).standard_normal((7, O)).astype(np.float32) * 10
        out = algo.policy(Batch(obs=obs, info=Batch()))
        assert out.act.shape == (7, A) and float(out.act.detach().abs().max()) <= max_action
        old = algo.policy(Batch(obs=obs, info=Batch()), model=algo.actor_old)
        assert torch.equal(old.act, out.act)                    # nothing trained yet: the lagged actor is the actor
        raw = out.act.detach().cpu().numpy()
        mapped = algo.policy.map_action(raw * 3)
        if bool(g["cfg_action_scaling"]):
            assert mapped.min() >= -1.0 and mapped.max() <= 1.0
        else:
            np.testing.assert_array_equal(mapped, raw * 3)       # action_bound_method=None, no scaling: unchanged
        assert isinstance(algo.policy.exploration_noise, GaussianNoise)
        np.random.seed(3)
        noisy = algo.policy.add_exploration_noise(raw, Batch(obs=obs))
        np.random.seed(3)
        np.testing.assert_array_equal(noisy, raw + np.random.normal(0.0, 0.1, raw.shape))
        algo.policy.set_exploration_noise(None)
        assert algo.policy.add_exploration_noise(raw, Batch(obs=obs)) is raw


def test_unsupported_actor_layer_is_refused():
    from tianshou_b200.algorithm import AdamOptimizerFactory, UnsupportedModelError
    from tianshou_b200.algorithm.modelfree.ddpg import ContinuousDeterministicPolicy
    from tianshou_b200.algorithm.modelfree.td3 import TD3
    from tianshou_b200.utils.net.common import Net
    from tianshou_b200.utils.net.continuous import ContinuousActorDeterministic, ContinuousCritic
    actor = ContinuousActorDeterministic(preprocess_net=Net(state_shape=(6,), hidden_sizes=(16,), activation=torch.nn.ELU),
                                         action_shape=(2,)).to(DEV)
    critic = ContinuousCritic(preprocess_net=Net(state_shape=(6,), action_shape=(2,), hidden_sizes=(16,), concat=True)).to(DEV)
    policy = ContinuousDeterministicPolicy(actor=actor, action_space=Box(2))
    with pytest.raises(UnsupportedModelError, match="actor.preprocess"):
        TD3(policy=policy, policy_optim=AdamOptimizerFactory(lr=1e-3), critic=critic, critic_optim=AdamOptimizerFactory(lr=1e-3))


def test_state_dict_round_trip():
    """Parameters, lagged copies and Adam moments survive ``state_dict()`` -> ``load_state_dict()`` into a fresh instance: the
    next update of both instances is the same."""
    from tianshou_b200.utils import policy_within_training_step
    g = load_golden("td3_ref.npz")
    algo, *_ = _build(g, True)
    buf = _buffer(g, True)
    for u in range(2):                      # update_actor_freq 2: the compared update below steps the actor
        torch.manual_seed(100 + u)
        with policy_within_training_step(algo.policy):
            algo.update(buffer=buf, sample_size=int(g["cfg_bs"]))
    sd = algo.state_dict()
    assert any(k.startswith("actor_old.") for k in sd) and any(k.startswith("critic2_old.") for k in sd)
    fresh, *_ = _build(g, True)
    with torch.no_grad():
        for p in fresh.parameters():
            p.mul_(0.5)
    fresh.load_state_dict(sd)
    fresh._cnt = algo._cnt                  # the delay counter is host state outside the state dict (as in the reference)
    for a, b in zip(algo._g_c + algo._g_ct + [algo._g_actor, algo._g_at], fresh._g_c + fresh._g_ct + [fresh._g_actor, fresh._g_at]):
        assert torch.equal(a.flat, b.flat)
    for a, b in zip(algo._g_c + [algo._g_actor], fresh._g_c + [fresh._g_actor]):
        assert torch.equal(a.exp_avg, b.exp_avg) and torch.equal(a.exp_avg_sq, b.exp_avg_sq) and a.step == b.step
    stats = []
    for x in (algo, fresh):                 # a buffer each, in the same state (the buffer's index RNG advances per update)
        torch.manual_seed(200)
        with policy_within_training_step(x.policy):
            stats.append(x.update(buffer=_buffer(g, True), sample_size=int(g["cfg_bs"])))
    assert _stat_losses(stats[0], True).tolist() == _stat_losses(stats[1], True).tolist()
    assert all(torch.equal(a.flat, b.flat) for a, b in zip(algo._g_c + [algo._g_actor], fresh._g_c + [fresh._g_actor]))
