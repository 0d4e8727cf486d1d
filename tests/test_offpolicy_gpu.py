"""Off-policy update bodies on the GPU (SURVEY 8(f) ranks 2-3) vs outputs of the imported reference
(tests/golden/sac_ref.npz, dqn_ref*.npz from oracle/gen_golden_offpolicy.py: same initial weights, same buffer contents,
same numpy / torch seeds): sampled indices bit-exact, n-step returns, losses, TD errors, post-update parameters of the
online and lagged networks."""
import numpy as np
import pytest
import torch

from ts_testutil import load_dqn_golden, load_golden, record_parity, set_buffer_state

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


class _Box:
    def __init__(self, dim):
        self.shape = (dim,)
        self.low = -np.ones(dim, np.float32)
        self.high = np.ones(dim, np.float32)


class _Discrete:
    def __init__(self, n):
        self.n = n
        self.shape = ()


def _load(mod, g, prefix):
    with torch.no_grad():
        for i, p in enumerate(mod.parameters()):
            p.copy_(torch.as_tensor(g[f"{prefix}{i}"]).reshape(p.shape))


def _check_params(tag, mod, g, prefix, lr):
    for i, p in enumerate(mod.parameters()):
        ref = g[f"{prefix}{i}"]
        # Adam normalises the step to ~lr per element: the absolute term is stated in units of one step
        record_parity(f"{tag}/{prefix}{i}", p.detach().cpu().numpy(), ref, rtol=1e-3, atol=0.1 * lr)


# ------------------------------------------------------------------------------------------------------------ SAC
def _build_sac(g, **kw):
    from tianshou_b200.algorithm import AdamOptimizerFactory
    from tianshou_b200.algorithm.modelfree.sac import SAC, SACPolicy
    from tianshou_b200.utils.net.common import Net
    from tianshou_b200.utils.net.continuous import ContinuousActorProbabilistic, ContinuousCritic
    O, A, H = int(g["cfg_obs"]), int(g["cfg_act"]), tuple(int(x) for x in g["cfg_hidden"])
    lr = float(g["cfg_lr"])
    actor = ContinuousActorProbabilistic(preprocess_net=Net(state_shape=(O,), hidden_sizes=H), action_shape=(A,), unbounded=True,
                                         conditioned_sigma=True).to(DEV)
    c1 = ContinuousCritic(preprocess_net=Net(state_shape=(O,), action_shape=(A,), hidden_sizes=H, concat=True)).to(DEV)
    c2 = ContinuousCritic(preprocess_net=Net(state_shape=(O,), action_shape=(A,), hidden_sizes=H, concat=True)).to(DEV)
    _load(actor, g, "p0_actor_"); _load(c1, g, "p0_c1_"); _load(c2, g, "p0_c2_")
    policy = SACPolicy(actor=actor, action_space=_Box(A))
    algo = SAC(policy=policy, policy_optim=AdamOptimizerFactory(lr=lr), critic=c1, critic_optim=AdamOptimizerFactory(lr=lr),
               critic2=c2, critic2_optim=AdamOptimizerFactory(lr=lr), tau=float(g["cfg_tau"]), gamma=float(g["cfg_gamma"]),
               alpha=float(g["cfg_alpha"]), n_step_return_horizon=int(g["cfg_n_step"]), **kw)
    return algo, actor, c1, c2, lr


@pytest.mark.parametrize("mirror", [False, True])
def test_sac_update_matches_reference(mirror):
    from tianshou_b200.data import Batch, VectorReplayBuffer
    from tianshou_b200.utils import policy_within_training_step
    g = load_golden("sac_ref.npz")
    algo, actor, c1, c2, lr = _build_sac(g)
    E, cap = int(g["cfg_E"]), int(g["cfg_cap"])
    buf = VectorReplayBuffer(E * cap, E, device=DEV, device_mirror=mirror)
    buf.set_batch(Batch(**{k: g["buf_" + k].copy() for k in ("obs", "act", "rew", "terminated", "truncated", "done", "obs_next")}))
    set_buffer_state(buf, g["meta_last_index"], g["meta_lengths"])
    if mirror:
        buf.sync_device_mirror()
        assert buf.device_columns() is not None
    # the reference drew its rsample noise from torch's CPU generator (it ran on the CPU): same draws, uploaded
    algo._noise_fn = lambda shape: torch.normal(torch.zeros(shape), torch.ones(shape)).to(DEV)
    captured = {}
    orig = algo._preprocess_batch

    def hook(batch, buffer, indices):
        b = orig(batch, buffer, indices)
        captured["indices"], captured["returns"] = np.asarray(indices).copy(), b.returns.detach().cpu().numpy().copy()
        return b

    algo._preprocess_batch = hook
    for u in range(int(g["cfg_updates"])):
        torch.manual_seed(100 + u)
        with policy_within_training_step(algo.policy):
            stats = algo.update(buffer=buf, sample_size=int(g["cfg_bs"]))
        o, tag = f"u{u}_", f"sac_m{int(mirror)}_u{u}"
        assert np.array_equal(captured["indices"], g[o + "indices"]), "sampled indices differ from the reference's"
        ref_ret = g[o + "returns"]
        record_parity(f"{tag}/returns", captured["returns"].reshape(ref_ret.shape), ref_ret, rtol=1e-5, atol=1e-5 * float(np.abs(ref_ret).max()))
        got = np.array([stats.actor_loss, stats.critic1_loss, stats.critic2_loss])
        record_parity(f"{tag}/losses", got, g[o + "losses"], rtol=2e-5, atol=2e-6)
        _check_params(tag, actor, g, o + "actor_", lr); _check_params(tag, c1, g, o + "c1_", lr); _check_params(tag, c2, g, o + "c2_", lr)
        _check_params(tag, algo.critic_old, g, o + "c1old_", lr); _check_params(tag, algo.critic2_old, g, o + "c2old_", lr)
        assert stats.alpha == pytest.approx(float(g["cfg_alpha"])) and stats.alpha_loss is None and stats.train_time > 0


def test_sac_cuda_graph_matches_reference():
    """``SAC(cuda_graph=True)``: update 0 runs eagerly, update 1 is captured and replayed, later updates are replays of the same
    graph — every one of them must still match the reference's update on the same indices / noise."""
    from tianshou_b200.data import Batch, VectorReplayBuffer
    from tianshou_b200.utils import policy_within_training_step
    g = load_golden("sac_ref.npz")
    algo, actor, c1, c2, lr = _build_sac(g, cuda_graph=True)
    E, cap = int(g["cfg_E"]), int(g["cfg_cap"])
    buf = VectorReplayBuffer(E * cap, E, device=DEV, device_mirror=True)
    buf.set_batch(Batch(**{k: g["buf_" + k].copy() for k in ("obs", "act", "rew", "terminated", "truncated", "done", "obs_next")}))
    set_buffer_state(buf, g["meta_last_index"], g["meta_lengths"])
    buf.sync_device_mirror()
    algo._noise_fn = lambda shape: torch.normal(torch.zeros(shape), torch.ones(shape)).to(DEV)
    n_up = int(g["cfg_updates"])
    assert n_up >= 3, "need an eager, a capture and a pure-replay update"
    for u in range(n_up):
        torch.manual_seed(100 + u)
        with policy_within_training_step(algo.policy):
            stats = algo.update(buffer=buf, sample_size=int(g["cfg_bs"]))
        o, tag = f"u{u}_", f"sac_graph_u{u}"
        assert np.array_equal(algo._graph["h_idx"].numpy(), g[o + "indices"]), "sampled indices differ from the reference's"
        got = np.array([stats.actor_loss, stats.critic1_loss, stats.critic2_loss])
        record_parity(f"{tag}/losses", got, g[o + "losses"], rtol=2e-5, atol=2e-6)
        _check_params(tag, actor, g, o + "actor_", lr); _check_params(tag, c1, g, o + "c1_", lr); _check_params(tag, c2, g, o + "c2_", lr)
        _check_params(tag, algo.critic_old, g, o + "c1old_", lr); _check_params(tag, algo.critic2_old, g, o + "c2old_", lr)
    assert algo._graph["graph"] is not None and algo._graph["calls"] == n_up
    for grp in algo._g_c:
        grp.sync_step_from_device()
        assert grp.step == n_up


def test_sac_policy_forward_collector_path():
    """``policy(batch)`` (the Collector's call, sac.py:108-131) keeps the Batch structure on the torch modules."""
    from tianshou_b200.data import Batch
    g = load_golden("sac_ref.npz")
    algo, actor, *_ = _build_sac(g)
    obs = np.random.default_rng(0).standard_normal((7, int(g["cfg_obs"]))).astype(np.float32)
    out = algo.policy(Batch(obs=obs, info=Batch()))
    assert out.act.shape == (7, int(g["cfg_act"])) and out.log_prob.shape == (7, 1) and float(out.act.abs().max()) <= 1.0
    assert algo.policy.map_action(out.act.detach().cpu().numpy()).shape == (7, int(g["cfg_act"]))


# ------------------------------------------------------------------------------------------------------------ DQN
def _build_dqn(g):
    from tianshou_b200.algorithm import AdamOptimizerFactory
    from tianshou_b200.algorithm.modelfree.dqn import DQN, DiscreteQLearningPolicy
    from tianshou_b200.env.atari import DQNet, ScaledObsInputActionReprNet
    H, W, A = int(g["cfg_H"]), int(g["cfg_W"]), int(g["cfg_A"])
    lr = float(g["cfg_lr"])
    net = ScaledObsInputActionReprNet(DQNet(4, H, W, A)).to(DEV)
    _load(net, g, "p0_q_")
    policy = DiscreteQLearningPolicy(model=net, action_space=_Discrete(A))
    huber = float(g["cfg_huber"])
    algo = DQN(policy=policy, optim=AdamOptimizerFactory(lr=lr), gamma=float(g["cfg_gamma"]), n_step_return_horizon=int(g["cfg_n_step"]),
               target_update_freq=int(g["cfg_target_freq"]), is_double=bool(g["cfg_is_double"]),
               huber_loss_delta=None if np.isnan(huber) else huber)
    return algo, net, lr


@pytest.mark.parametrize("variant,mirror", [("", True), ("", False), ("_b", True)])
def test_dqn_update_matches_reference(variant, mirror):
    """NatureCNN DQN on uint8 single-frame storage (stack_num 4, save_only_last_obs, ignore_obs_next) with prioritised
    replay: the frame stacks are gathered by the first convolution's im2col from the device copy of the frames."""
    from tianshou_b200.data import Batch, PrioritizedVectorReplayBuffer
    from tianshou_b200.utils import policy_within_training_step
    g = load_dqn_golden(variant)
    algo, net, lr = _build_dqn(g)
    E, cap, steps = int(g["cfg_E"]), int(g["cfg_cap"]), int(g["cfg_steps"])
    buf = PrioritizedVectorReplayBuffer(E * cap, E, alpha=float(g["cfg_alpha"]), beta=float(g["cfg_beta"]), stack_num=4,
                                        ignore_obs_next=True, save_only_last_obs=True, device=DEV, device_mirror=mirror)
    for i in range(steps):
        last = g[f"roll{i}_obs"]
        stack = np.repeat(last[:, None], 4, axis=1)            # only the last frame is stored (save_only_last_obs)
        buf.add(Batch(obs=stack, act=g[f"roll{i}_act"], rew=g[f"roll{i}_rew"], terminated=g[f"roll{i}_terminated"],
                      truncated=g[f"roll{i}_truncated"], obs_next=stack), buffer_ids=np.arange(E))
    assert buf.obs.dtype == np.uint8 and buf.obs.shape[1:] == (int(g["cfg_H"]), int(g["cfg_W"]))
    if mirror:
        assert buf.device_columns() is not None and buf.device_columns()["obs"].dtype == torch.uint8
    captured = {}
    orig_pre, orig_post = algo._preprocess_batch, algo._postprocess_batch

    def pre(batch, buffer, indices):
        captured["is_weight"] = batch.weight.detach().cpu().numpy().copy()
        b = orig_pre(batch, buffer, indices)
        captured["indices"], captured["returns"] = np.asarray(indices).copy(), b.returns.detach().cpu().numpy().copy()
        return b

    def post(batch, buffer, indices):
        captured["td"] = batch.weight.detach().cpu().numpy().copy()
        return orig_post(batch, buffer, indices)

    algo._preprocess_batch, algo._postprocess_batch = pre, post
    n_up = int(g["cfg_updates"])
    for u in range(n_up):
        np.random.seed(500 + u)
        with policy_within_training_step(algo.policy):
            stats = algo.update(buffer=buf, sample_size=int(g["cfg_bs"]))
        o, tag = f"u{u}_", f"dqn{variant}_m{int(mirror)}_u{u}"
        assert np.array_equal(captured["indices"], g[o + "indices"]), f"update {u}: sampled indices differ from the reference's"
        record_parity(f"{tag}/is_weight", captured["is_weight"], g[o + "is_weight"], rtol=1e-4, atol=1e-6)
        ref_ret = g[o + "returns"]
        record_parity(f"{tag}/returns", captured["returns"].reshape(ref_ret.shape), ref_ret, rtol=1e-5, atol=1e-5 * float(np.abs(ref_ret).max()))
        record_parity(f"{tag}/td", captured["td"], g[o + "td"], rtol=1e-5, atol=2e-5 * float(np.abs(g[o + "td"]).max()))
        record_parity(f"{tag}/loss", np.array([stats.loss]), np.array([float(g[o + "loss"])]), rtol=2e-5, atol=1e-6)
        record_parity(f"{tag}/tree_leaves", np.asarray(buf.weight[np.arange(len(buf))]), g[o + "tree_leaves"], rtol=1e-4, atol=1e-7)
    o = f"u{n_up - 1}_"
    _check_params(f"dqn{variant}_m{int(mirror)}", net, g, o + "q_", lr)
    if algo.model_old is not None:
        _check_params(f"dqn{variant}_m{int(mirror)}", algo.model_old, g, o + "qold_", lr)


def test_dqn_policy_forward_and_eps_greedy():
    from tianshou_b200.data import Batch
    g = load_golden("dqn_ref_b.npz")
    algo, net, _ = _build_dqn(g)
    obs = np.random.default_rng(0).integers(0, 256, (5, 4, int(g["cfg_H"]), int(g["cfg_W"])), dtype=np.uint8)
    out = algo.policy(Batch(obs=obs, info=Batch()))
    assert out.logits.shape == (5, int(g["cfg_A"])) and out.act.shape == (5,)
    algo.policy.set_eps_inference(1.0)
    np.random.seed(0)
    act = algo.policy.add_exploration_noise(out.act.copy(), Batch(obs=obs))
    assert act.shape == (5,) and act.min() >= 0 and act.max() < int(g["cfg_A"])
