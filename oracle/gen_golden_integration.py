"""TEST INFRASTRUCTURE -- golden call trace of the UNMODIFIED reference ``Collector`` + ``OnPolicyTrainer`` (thu-ml/tianshou
2.0.1, imported through oracle/ref_shim.py) driving this package's ``VectorReplayBuffer`` / ``DiscreteActorPolicy`` /
``OnPolicyAlgorithm`` (BASELINE configs[0]: 10 CartPole-shaped envs, two epochs).

    python -m oracle.gen_golden_integration        # writes tests/golden/integration_ref.npz

Recorded, in call order: every ``buffer.add`` (the Collector's rows, buffer ids and what ``add`` returned, stacked over
the calls), every ``buffer.reset``, every ``algorithm.update`` (arguments, numpy's global generator state and the learning
rate at entry; mean loss and learning rate after it), plus the parameters before the first and after the last update.  tests/test_integration_reference.py
replays the sequence without the reference and compares.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
OUT = os.path.join(ROOT, "tests", "golden")

from oracle.ref_shim import import_reference  # noqa: E402

ts = import_reference()
import gymnasium as gym  # noqa: E402  (the shim's stand-in spaces)
import tianshou.data.collector as refcol  # noqa: E402
from tianshou.env import DummyVectorEnv  # noqa: E402
from tianshou.trainer import OnPolicyTrainer, OnPolicyTrainerParams  # noqa: E402

import tianshou_b200.compat as compat  # noqa: E402
from test_integration_reference import ADD_KEYS, E, build_oracle_ppo, params_of  # noqa: E402
from tianshou_b200.data import VectorReplayBuffer  # noqa: E402


class FakeCartPole:
    """CartPole-shaped stand-in (gymnasium is not installed): obs 4, 2 actions, reward 1 per step."""

    metadata: dict = {}
    spec = None

    def __init__(self, seed: int = 0):
        self.action_space = gym.spaces.Discrete(2)
        self.observation_space = gym.spaces.Box(-1.0, 1.0, (4,))
        self.rng = np.random.default_rng(seed)
        self.t = 0
        self.unwrapped = self

    def reset(self, seed=None, options=None):
        self.t = 0
        return self.rng.standard_normal(4).astype(np.float32), {}

    def step(self, a):
        self.t += 1
        term = bool(self.rng.random() < 0.05)
        return self.rng.standard_normal(4).astype(np.float32), 1.0, term, self.t >= 30 and not term, {}

    def close(self):
        pass

    def seed(self, s=None):
        return [s]

    def render(self):
        return None


def main() -> None:
    compat.install_into_reference()
    torch.manual_seed(0)
    np.random.seed(0)
    algo, actor, critic = build_oracle_ppo(gym.spaces.Discrete(2))
    out: dict[str, np.ndarray] = {f"p0_{k}": v.detach().numpy().copy() for k, v in params_of(actor, critic).items()}
    buf = VectorReplayBuffer(E * 40, E)
    events: list[int] = []                 # 0 = add, 1 = reset, 2 = update
    adds: dict[str, list[np.ndarray]] = {}    # one row per add() call (the Collector adds one step of every env at a time)
    n = {"reset": 0, "update": 0}
    add, reset, update = buf.add, buf.reset, algo.update

    def rec_add(batch, buffer_ids=None):
        for k in ADD_KEYS:
            adds.setdefault(k, []).append(np.asarray(getattr(batch, k)).copy())
        adds.setdefault("buffer_ids", []).append(np.asarray(buffer_ids, dtype=np.int64).copy())
        ret = add(batch, buffer_ids=buffer_ids)
        for k, r in zip(("ptr", "ep_rew", "ep_len", "ep_idx"), ret, strict=True):
            adds.setdefault("ret_" + k, []).append(np.asarray(r).copy())
        events.append(0)
        return ret

    def rec_reset(keep_statistics=False):
        out[f"reset{n['reset']}_keep_statistics"] = np.asarray(bool(keep_statistics))
        events.append(1)
        n["reset"] += 1
        return reset(keep_statistics=keep_statistics)

    def rec_update(buffer, batch_size, repeat):
        assert buffer is buf
        o = f"update{n['update']}_"
        st = np.random.get_state()
        out[o + "np_key"], out[o + "np_pos"] = np.asarray(st[1], dtype=np.uint32).copy(), np.asarray(st[2], dtype=np.int64)
        out[o + "batch_size"], out[o + "repeat"] = np.asarray(batch_size, dtype=np.int64), np.asarray(repeat, dtype=np.int64)
        out[o + "lr_before"] = np.asarray(algo.optim._optim.param_groups[0]["lr"], dtype=np.float64)
        stats = update(buffer, batch_size, repeat)
        out[o + "loss_mean"] = np.asarray(stats.loss.mean, dtype=np.float64)
        out[o + "gradient_steps"] = np.asarray(stats.gradient_steps, dtype=np.int64)
        out[o + "lr_after"] = np.asarray(algo.optim._optim.param_groups[0]["lr"], dtype=np.float64)
        out[o + "rows"] = np.asarray(algo.calls[-1][0], dtype=np.int64)
        for k, v in params_of(actor, critic).items():      # overwritten: the parameters after the LAST update are kept
            out["final_p_" + k] = v.detach().numpy().copy()
        events.append(2)
        n["update"] += 1
        return stats

    buf.add, buf.reset, algo.update = rec_add, rec_reset, rec_update
    envs = DummyVectorEnv([lambda i=i: FakeCartPole(i) for i in range(E)])
    collector = refcol.Collector(algo, envs, buf)
    params = OnPolicyTrainerParams(training_collector=collector, test_collector=None, max_epochs=2, epoch_num_steps=400,
                                   collection_step_num_env_steps=200, batch_size=64, update_step_num_repetitions=2,
                                   test_in_training=False, verbose=False, show_progress=False)
    OnPolicyTrainer(algo, params).run()
    out["events"] = np.asarray(events, dtype=np.int8)
    out.update({"add_" + k: np.stack(v) for k, v in adds.items()})
    np.savez_compressed(os.path.join(OUT, "integration_ref.npz"), **out)
    print("integration_ref.npz", len(out), "arrays;", n)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    main()
