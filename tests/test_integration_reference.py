"""BASELINE configs[0] plumbing: the UNMODIFIED reference ``Collector`` + ``OnPolicyTrainer`` drive this package's
``Batch`` / ``VectorReplayBuffer`` / ``DiscreteActorPolicy`` / ``OnPolicyAlgorithm`` on a 10-env CartPole-shaped
environment for two epochs.

tests/golden/integration_ref.npz (oracle/gen_golden_integration.py) is the call trace of that run: every ``buffer.add``
the reference Collector made (its rows, buffer ids and what ``add`` returned), every ``buffer.reset`` of the trainer's
``reset_buffer``, every ``algorithm.update`` the trainer made (arguments, numpy's generator state and learning rate at
entry; mean loss and learning rate after it, parameters after the last one).  The test replays that sequence on fresh objects and checks that
they return and compute what they did under the reference.  The numeric body of ``_update_with_batch`` is the numpy
oracle (CPU test) -- everything AROUND it is the product: ``buffer.add`` of the Collector's rows (collector.py:927-930),
``reset_buffer`` (trainer.py:1131), ``Algorithm.update`` with its training-step guard and lr scheduler
(algorithm_base.py:586-631), the stats dataclass the trainer serialises (trainer.py:733-737,1122), and the
``tianshou_b200.compat`` widening of the collector's ``isinstance`` gates (collector.py:360,375-384).
"""
import dataclasses
import types

import numpy as np
import pytest
import torch

from ts_testutil import load_golden

E = 10
ADD_KEYS = ("obs", "act", "rew", "terminated", "truncated", "obs_next")


def params_of(actor, critic) -> dict:
    """Every parameter of the shared-trunk actor / critic pair, by the numpy oracle's names."""
    t1, t2 = [m for m in actor.preprocess.model.model if isinstance(m, torch.nn.Linear)]
    a3, c3 = actor.last.model[0], critic.last.model[0]
    return {"a_w1": t1.weight, "a_b1": t1.bias, "a_w2": t2.weight, "a_b2": t2.bias, "a_w3": a3.weight, "a_b3": a3.bias,
            "c_w3": c3.weight, "c_b3": c3.bias}


def build_oracle_ppo(action_space):
    """This package's ``OnPolicyAlgorithm`` skeleton around a ``DiscreteActorPolicy``, with the numeric body of the update
    from the numpy oracle (CPU stand-in for the kernels)."""
    from oracle import oracle_discrete as od
    from oracle import oracle_np as onp
    from tianshou_b200.algorithm import A2CTrainingStats, AdamOptimizerFactory, DiscreteActorPolicy, OnPolicyAlgorithm
    from tianshou_b200.algorithm.optim import LRSchedulerFactoryLinear
    from tianshou_b200.data import Batch, SequenceSummaryStats, VectorReplayBuffer
    from tianshou_b200.utils.net.common import ActorCritic, Net
    from tianshou_b200.utils.net.discrete import DiscreteActor, DiscreteCritic

    net = Net(state_shape=(4,), hidden_sizes=(64, 64))
    actor = DiscreteActor(preprocess_net=net, action_shape=2, softmax_output=True)
    critic = DiscreteCritic(preprocess_net=net)
    policy = DiscreteActorPolicy(actor=actor, dist_fn=lambda p: torch.distributions.Categorical(probs=p),
                                 action_space=action_space)

    class OraclePPO(OnPolicyAlgorithm):
        def __init__(self):
            super().__init__(policy=policy)
            self.critic = critic
            self.optim = self._create_optimizer(ActorCritic(actor, critic), AdamOptimizerFactory(lr=3e-4).with_lr_scheduler_factory(
                LRSchedulerFactoryLinear(max_epochs=2, epoch_num_steps=400, collection_step_num_env_steps=200)))
            self.calls, self.rms = [], onp.RunningMeanStd()
            self.m = self.v = None
            self.step = 0

        def _sample(self, buffer, sample_size):
            assert sample_size == 0 and isinstance(buffer, VectorReplayBuffer)
            idx = np.concatenate([np.arange(e * buffer._cap[e], e * buffer._cap[e] + buffer._sizes[e]) for e in range(E)])
            return buffer._meta[idx], idx                # un-wrapped sub-buffers: chronological order per env

        def _update_with_batch(self, batch, batch_size, repeat):
            assert self.policy.is_within_training_step and isinstance(batch, Batch)
            self.calls.append((len(batch), batch_size, repeat))
            tp = params_of(actor, critic)
            p = {k: v.detach().numpy().copy() for k, v in tp.items()}
            if self.m is None:
                self.m = {k: np.zeros_like(v) for k, v in p.items()}
                self.v = {k: np.zeros_like(v) for k, v in p.items()}
            n = len(batch)
            done = np.asarray(batch.terminated) | np.asarray(batch.truncated)
            unf = np.zeros(n, bool)
            ends = np.cumsum([self._last_sizes[e] for e in range(E)]) - 1
            unf[ends] = ~done[ends]
            roll = dict(obs=np.asarray(batch.obs, np.float32), obs_next=np.asarray(batch.obs_next, np.float32), act=np.asarray(batch.act),
                        rew=np.asarray(batch.rew, np.float64), terminated=np.asarray(batch.terminated), truncated=np.asarray(batch.truncated),
                        unfinished=unf)
            perms = [np.random.permutation(n) for _ in range(repeat)]
            hp = dict(eps_clip=0.2, dual_clip=None, vf_coef=0.5, ent_coef=0.0, max_grad_norm=0.5, adv_eps=1e-8, value_clip=False,
                      advantage_normalization=True, lr=self.optim._optim.param_groups[0]["lr"], beta1=0.9, beta2=0.999, adam_eps=1e-8,
                      weight_decay=0.0)
            res = od.ppo_update(p, self.m, self.v, self.step, roll, perms, batch_size, repeat, hp, None, 0.99, 0.95, False)
            self.step = res["step"]
            with torch.no_grad():
                for k, t in tp.items():
                    t.copy_(torch.from_numpy(p[k]))
            ls = res["losses"]
            return A2CTrainingStats(loss=SequenceSummaryStats.from_sequence(ls[:, 0]), actor_loss=SequenceSummaryStats.from_sequence(ls[:, 1]),
                                    vf_loss=SequenceSummaryStats.from_sequence(ls[:, 2]), ent_loss=SequenceSummaryStats.from_sequence(ls[:, 3]),
                                    gradient_steps=len(ls))

        def update(self, buffer, batch_size, repeat):
            self._last_sizes = buffer._sizes.copy()
            return super().update(buffer, batch_size, repeat)

    return OraclePPO(), actor, critic


def test_compat_widens_the_collector_gates():
    import tianshou_b200.compat as compat
    from tianshou_b200.algorithm.base import Algorithm
    from tianshou_b200.data import ReplayBufferManager

    class RefAlgorithm:                                  # the reference collector module's own names
        pass

    class RefReplayBufferManager:
        pass

    mod = types.SimpleNamespace(Algorithm=RefAlgorithm, ReplayBufferManager=RefReplayBufferManager)
    compat.install_into_reference(mod)
    compat.install_into_reference(mod)                   # idempotent
    assert mod.Algorithm == (RefAlgorithm, Algorithm)
    assert mod.ReplayBufferManager == (RefReplayBufferManager, ReplayBufferManager)


def test_reference_collector_and_trainer_drive_b200_types():
    from tianshou_b200.data import Batch, VectorReplayBuffer
    from tianshou_b200.utils import policy_within_training_step

    g = load_golden("integration_ref.npz")
    algo, actor, critic = build_oracle_ppo(types.SimpleNamespace(n=2, shape=()))
    with torch.no_grad():
        for k, t in params_of(actor, critic).items():
            t.copy_(torch.from_numpy(g["p0_" + k]))
    buf = VectorReplayBuffer(E * 40, E)
    w0 = actor.last.model[0].weight.detach().clone()
    with pytest.raises(RuntimeError):                                       # update outside a training step (algorithm_base.py:612-617)
        algo.update(buf, 64, 1)
    n_add = n_reset = n_update = 0
    for ev in g["events"]:
        if ev == 0:
            ret = buf.add(Batch(**{k: g["add_" + k][n_add] for k in ADD_KEYS}), buffer_ids=g["add_buffer_ids"][n_add])
            for k, r in zip(("ptr", "ep_rew", "ep_len", "ep_idx"), ret, strict=True):
                np.testing.assert_array_equal(np.asarray(r), g["add_ret_" + k][n_add], err_msg=f"add {n_add}: {k}")
            n_add += 1
        elif ev == 1:
            buf.reset(keep_statistics=bool(g[f"reset{n_reset}_keep_statistics"]))
            n_reset += 1
        else:
            o = f"update{n_update}_"
            np.random.set_state(("MT19937", g[o + "np_key"], int(g[o + "np_pos"]), 0, 0.0))
            assert algo.optim._optim.param_groups[0]["lr"] == float(g[o + "lr_before"])
            with policy_within_training_step(algo.policy):
                stats = algo.update(buf, int(g[o + "batch_size"]), int(g[o + "repeat"]))
            assert algo.calls[-1][0] == int(g[o + "rows"])
            assert stats.gradient_steps == int(g[o + "gradient_steps"])
            np.testing.assert_allclose(stats.loss.mean, float(g[o + "loss_mean"]), rtol=1e-12, atol=1e-12)
            np.testing.assert_allclose(algo.optim._optim.param_groups[0]["lr"], float(g[o + "lr_after"]), rtol=1e-12)
            assert isinstance(dataclasses.asdict(stats), dict)
            n_update += 1
    assert n_add > 0 and n_reset > 0
    for k, t in params_of(actor, critic).items():
        np.testing.assert_allclose(t.detach().numpy(), g["final_p_" + k], rtol=1e-6, atol=1e-7, err_msg=k)
    assert len(algo.calls) == 4 and all(c[1:] == (64, 2) for c in algo.calls)          # 2 epochs x (400 / 200) update steps
    assert all(c[0] == 200 for c in algo.calls), algo.calls                             # the buffer was reset between collects
    assert not torch.equal(w0, actor.last.model[0].weight)                              # parameters moved
    assert algo.optim._optim.param_groups[0]["lr"] < 3e-4                               # lr scheduler stepped once per update()
    assert len(buf) <= E * 40
