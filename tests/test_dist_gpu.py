"""Multi-GPU path (one process per GPU): with identical rollouts on both ranks the averaged gradient
equals the single-GPU gradient, so the update must reproduce the reference run -- both through the fused
kernel (gradient sum inside the persistent epoch kernel over NVLink peer memory, ``path="p2p"``) and
through the per-step NCCL all-reduce (``path="nccl"``)."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port() -> int:
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank: int, world_size: int, port: int, variant: str, path: str, out_dir: str, partition: str = "per_rank") -> None:
    import torch.distributed as dist

    from test_ppo_gpu import ppo_kwargs
    from tianshou_b200.utils import policy_within_training_step
    from ts_testutil import PARAM_ORDER, build_ppo, load_golden, named_params, restore_vector_buffer

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size),
                      TS_B200_NO_P2P="1" if path == "nccl" else "0")
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world_size, device_id=dev)
    try:
        g = load_golden(f"ppo_ref_{variant}.npz")
        kw = ppo_kwargs(g)
        lr = float(g["kw_lr"]) if "kw_lr" in g.files else 3e-4
        algo, actor, critic = build_ppo(17, 6, dev, lr=lr, params={k: g["p0_" + k] for k in PARAM_ORDER},
                                        rollout_partition=partition, **kw)
        bs = int(g["cfg_bs"])
        for u in range(2):
            buf = restore_vector_buffer(g, f"u{u}_", int(g["cfg_E"]), int(g["cfg_cap"]), device=dev)
            np.random.seed(1000 + u)
            with policy_within_training_step(algo.policy):
                stats = algo.update(buffer=buf, batch_size=None if bs < 0 else bs, repeat=int(g["cfg_repeat"]))
            assert stats.gradient_steps == int(g[f"u{u}_gradient_steps"])
            # the path under test is the one that ran (no silent fallback)
            assert (algo._scratch.get("peer_exchange") is not None) == (path == "p2p"), "wrong multi-GPU path"
            ref_losses = g[f"u{u}_losses"]
            np.testing.assert_allclose(stats.loss.mean, ref_losses[:, 0].mean(), rtol=5e-4, atol=2e-5)
            np.testing.assert_allclose(stats.vf_loss.mean, ref_losses[:, 2].mean(), rtol=5e-4, atol=2e-5)
            for k, pv in named_params(actor, critic).items():
                np.testing.assert_allclose(pv.detach().cpu().numpy(), g[f"u{u}_p_" + k], rtol=2e-3, atol=3e-5,
                                           err_msg=f"rank {rank} update {u} {k}")
            if kw["return_scaling"]:   # two identical shards: same mean / var, twice the count (shared rollout: the count too)
                np.testing.assert_allclose([algo.ret_rms.mean, algo.ret_rms.var], g[f"u{u}_rms"][:2], rtol=1e-5)
                if partition == "shared":
                    np.testing.assert_allclose(algo.ret_rms.count, g[f"u{u}_rms"][2], rtol=1e-12)
            if partition == "shared":  # the SAME problem as the reference run: the per-minibatch loss table must match row by row
                np.testing.assert_allclose(algo.last_loss_table[:, :4], ref_losses, rtol=2e-4, atol=2e-5)
        torch.save(algo._flat.flat.cpu(), os.path.join(out_dir, f"flat{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("path", ["p2p", "nccl"])
@pytest.mark.parametrize("variant", ["A", "B"])
def test_two_rank_update_matches_reference(variant, path, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), variant, path, str(tmp_path)), nprocs=2, join=True)
    a, b = torch.load(tmp_path / "flat0.pt"), torch.load(tmp_path / "flat1.pt")
    assert torch.equal(a, b), "replicas diverged"      # same all-reduced gradient, same Adam step: bit-identical


@pytest.mark.parametrize("variant", ["A", "B"])
def test_two_rank_shared_rollout_matches_reference(variant, tmp_path):
    """Strong scaling (SURVEY 8(e)): ONE rollout, the same ``np.random.permutation`` stream on both ranks, every minibatch split
    into two contiguous slices, gradient sum inside the epoch kernel -> the reference run's results, loss table row by row.
    Variant B's golden uses a minibatch size that does not divide the rollout (ragged last minibatch): a shared rollout
    refuses that split loudly (``ValueError`` from ``PPO._shared_slice``) instead of changing the minibatch composition."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    if variant == "B":
        with pytest.raises(Exception, match="rollout_partition='shared' needs"):
            mp.spawn(_worker, args=(2, _free_port(), variant, "p2p", str(tmp_path), "shared"), nprocs=2, join=True)
        return
    mp.spawn(_worker, args=(2, _free_port(), variant, "p2p", str(tmp_path), "shared"), nprocs=2, join=True)
    a, b = torch.load(tmp_path / "flat0.pt"), torch.load(tmp_path / "flat1.pt")
    assert torch.equal(a, b), "replicas diverged"
