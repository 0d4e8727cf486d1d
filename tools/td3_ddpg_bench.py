"""ms per ``update()`` of TD3 and DDPG on a Humanoid-shaped workload (obs 376, act 17, MLP[256, 256], batch 256,
update_actor_freq 2, a 64 x 1024 transition buffer with a device mirror, 1 GPU), eager and ``cuda_graph=True``, next to the
torch-CPU port and the same torch code run as stock eager PyTorch on the same GPU (oracle/oracle_det.py; a context
number: it gathers rows and computes n-step returns on the host as the reference does).  Prints one JSON line.

    python tools/td3_ddpg_bench.py [--updates 200] [--repeats 3] [--out FILE]

Each of the four device variants warms up 8 updates first (TD3: both graphs are captured by then), then the timed windows
alternate between the variants ``--repeats`` times; median / min / max over the windows are reported.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

O, A, H, B, E, STEPS, FREQ, LR = 376, 17, (256, 256), 256, 64, 1024, 2, 1e-3


def gpu_info() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        pl, mhz = (x.strip() for x in r.stdout.strip().split(","))
        info.update(power_limit_w=float(pl), sm_max_mhz=float(mhz))
    except Exception as ex:  # noqa: BLE001
        info["power_limit_w"] = f"unavailable: {ex!r}"
    return info


def stats(xs: list[float]) -> dict:
    return {"median": float(np.median(xs)), "min": float(min(xs)), "max": float(max(xs)), "n": len(xs)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--updates", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--cpu-updates", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU path; there is no CPU fallback"
    assert args.warmup >= 6, "at least 6 warm-up updates: both TD3 graphs must be captured before timing"
    from oracle import oracle_det as od
    from tianshou_b200.algorithm import AdamOptimizerFactory
    from tianshou_b200.algorithm.modelfree.ddpg import DDPG, ContinuousDeterministicPolicy
    from tianshou_b200.algorithm.modelfree.td3 import TD3
    from tianshou_b200.data import Batch, VectorReplayBuffer
    from tianshou_b200.synthetic import BoxSpace
    from tianshou_b200.utils import policy_within_training_step
    from tianshou_b200.utils.net.common import Net
    from tianshou_b200.utils.net.continuous import ContinuousActorDeterministic, ContinuousCritic

    dev = torch.device("cuda:0")
    gpu = gpu_info()
    rng = np.random.default_rng(0)
    buf = VectorReplayBuffer(E * STEPS, E, device=dev, device_mirror=True)
    obs = rng.standard_normal((E, O)).astype(np.float32)
    for _ in range(STEPS):
        nxt = rng.standard_normal((E, O)).astype(np.float32)
        buf.add(Batch(obs=obs, act=np.tanh(rng.standard_normal((E, A))).astype(np.float32), rew=rng.standard_normal(E),
                      terminated=rng.random(E) < 1e-3, truncated=np.zeros(E, bool), obs_next=nxt), buffer_ids=np.arange(E))
        obs = nxt

    torch.manual_seed(0)
    actor = ContinuousActorDeterministic(preprocess_net=Net(state_shape=(O,), hidden_sizes=H), action_shape=(A,)).to(dev)
    critics = [ContinuousCritic(preprocess_net=Net(state_shape=(O,), action_shape=(A,), hidden_sizes=H, concat=True)).to(dev)
               for _ in range(2)]

    def make(kind: str, graph: bool):
        a, c1, c2 = copy.deepcopy((actor, *critics))
        kw = dict(policy=ContinuousDeterministicPolicy(actor=a, action_space=BoxSpace(A)), policy_optim=AdamOptimizerFactory(lr=LR),
                  critic=c1, critic_optim=AdamOptimizerFactory(lr=LR), tau=0.005, gamma=0.99, cuda_graph=graph)
        if kind == "td3":
            return TD3(critic2=c2, critic2_optim=AdamOptimizerFactory(lr=LR), update_actor_freq=FREQ, **kw)
        return DDPG(**kw)

    variants = {(k, g): make(k, g) for k in ("td3", "ddpg") for g in (False, True)}

    def run(algo, n: int) -> float:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with policy_within_training_step(algo.policy):
            for _ in range(n):
                algo.update(buffer=buf, sample_size=B)
        torch.cuda.synchronize()
        return 1e3 * (time.perf_counter() - t0) / n

    for algo in variants.values():
        run(algo, args.warmup)
    times: dict = {v: [] for v in variants}
    for _ in range(args.repeats):                      # alternate the variants: drift on a shared host hits all of them
        for v, algo in variants.items():
            times[v].append(run(algo, args.updates))
    replaying = {k: all(x["graph"] is not None for x in variants[(k, True)]._graphs.values()) for k in ("td3", "ddpg")}
    n_graphs = {k: len(variants[(k, True)]._graphs) for k in ("td3", "ddpg")}
    del variants

    # the same update as plain torch code: on the CPU (the port) and as eager PyTorch on this GPU (context)
    host = dict(obs=np.asarray(buf.obs), act=np.asarray(buf.act), rew=np.asarray(buf.rew), done=np.asarray(buf.done),
                terminated=np.asarray(buf.terminated), obs_next=np.asarray(buf.obs_next), offset=np.asarray(buf._extend_offset),
                last_index=np.asarray(buf.last_index), lengths=np.asarray(buf._sizes))
    cpu_threads = min(8, os.cpu_count() or 1)
    torch.set_num_threads(cpu_threads)

    def torch_ms(kind: str, device: str, n: int, warm: int) -> float:
        nets = od.DetNets(O, A, H, 2 if kind == "td3" else 1, device=device)
        opts = [torch.optim.Adam(nets.actor.parameters(), lr=LR)] + [torch.optim.Adam(c.parameters(), lr=LR) for c in nets.c]
        cnt = 0

        def one():
            nonlocal cnt
            idx = rng.integers(0, E * STEPS, B)
            if kind == "td3":
                od.td3_update(nets, opts, host, idx, torch.randn(B, A, device=device), 0.2, 0.5, 0.99, 1, 0.005, cnt % FREQ == 0)
            else:
                od.ddpg_update(nets, opts, host, idx, 0.99, 1, 0.005)
            cnt += 1
        for _ in range(warm):
            one()
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n):
            one()
        if device != "cpu":
            torch.cuda.synchronize()
        return 1e3 * (time.perf_counter() - t0) / n

    out: dict = {"gpu": gpu, "workload": f"update(sample_size={B}) obs {O} act {A} MLP{list(H)}, TD3 update_actor_freq {FREQ}, "
                 f"VectorReplayBuffer {E}x{STEPS} transitions with device mirror, n_step 1, 1 GPU",
                 "timed_updates_per_window": args.updates, "warmup_updates": args.warmup}
    for kind in ("td3", "ddpg"):
        eager = [torch_ms(kind, "cuda:0", args.updates // 2, 6) for _ in range(args.repeats)]
        out[kind] = {
            "ms_per_update": stats(times[(kind, False)]),
            "cuda_graph": {"ms_per_update": stats(times[(kind, True)]), "replaying": replaying[kind], "graphs": n_graphs[kind]},
            "torch_eager_gpu": {"ms_per_update": stats(eager),
                                "kind": "context: oracle/oracle_det.py as stock eager PyTorch on this GPU (host n-step)"},
            "cpu_port": {"ms_per_update": torch_ms(kind, "cpu", args.cpu_updates, 2), "threads": torch.get_num_threads(),
                         "kind": "port (torch CPU, oracle/oracle_det.py)"},
        }
    out["gpu_after"] = gpu_info()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
