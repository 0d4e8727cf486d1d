#!/usr/bin/env python
"""bench.py -- transitions/sec through PPO ``Algorithm.update()`` (v1: ``learn()``), obs=17.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config c2|c5] [--scaling weak|strong]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1], SURVEY.md 8d): synthetic HalfCheetah-shaped rollout of
4096 envs x 128 steps per GPU (N = 524,288 transitions, obs 17, act 6), actor/critic MLP[64,64]
tanh, hyper-parameters of examples/mujoco/mujoco_ppo.py (gamma .99, lambda .95, eps .2, vf .25,
ent 0, max_grad_norm .5, value_clip, recompute_advantage, return_scaling, Adam 3e-4),
minibatch 16384, repeat 10  ->  320 optimiser steps + 10 value/GAE passes per update.
A "step" of this benchmark is ONE ``update(buffer, batch_size=16384, repeat=10)`` call.

Reported (one JSON line on rank 0):
  value : transitions/s with the rollout already resident in HBM (device preprocess + update).
  e2e   : transitions/s through the public API ``PPO.update(buffer, ...)`` with the rollout in
          (pinned) host buffers: bulk H2D of the rollout and D2H of the loss table inside the
          timed region.
  roofline : dominant kernel (minibatch forward/backward) against the measured bf16 GEMM peak,
             algorithmic flops 60,544 / row (SURVEY.md 8d).
  cpu_baseline / --impl reference : the numpy port of the reference's update (oracle/) timed on
             this box's host cores on a bounded sample of the same workload.
Multi-GPU (torchrun): default = weak scaling -- every rank owns its own 4096x128 rollout shard, the global
minibatch is N x 16384 rows, the gradient sum over the ranks happens INSIDE the persistent epoch kernel (8-byte
packets over NVLink peer memory); value = all ranks' transitions / max-over-ranks time.  ``--scaling strong``: ONE
rollout replicated on every rank, the same host permutation, each minibatch split into N contiguous slices (SURVEY
8(e)): a fixed problem whose results equal the single-GPU run's.  Outside the timed region every multi-GPU run also
checks itself: ``multi_gpu_check`` = {replicas_equal, loss_rel_err (N ranks vs 1 rank on the same inputs), ...}.
``--config c5`` = BASELINE configs[4] (8192 envs x 256 steps, minibatch N/8); the default run reports it as the extra
key ``config4`` (strong-scaled over the N GPUs).  The timed arms use the DEFAULT public API (reference-exact
``np.random.permutation`` minibatch order); the opt-in device-generated order is reported as ``*_device_order``.
``--dump-outputs DIR`` writes what the last timed step of the headline arm computed (see ``dump_outputs``): the inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

OBS, ACT = 17, 6
E_FULL, T_FULL = 4096, 128
BATCH_SIZE, REPEAT = 16384, 10
FLOP_TRAIN_PER_ROW = 60_544          # fwd+bwd of actor and critic (SURVEY 8d)
FLOP_PER_TRANSITION = REPEAT * 81_536 + 11_136
METRIC = "transitions/sec through Algorithm.learn() (PPO, obs=17)"
DUMP_ROWS = 1 << 20                  # per-transition outputs of longer rollouts are dumped as a fixed seeded sample of rows
DUMP_BYTES = 64 << 20


def load_peaks() -> tuple[dict, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows: list[list[str]] = []
        self.proc = None
        self.gpu = gpu_index
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
        except OSError:
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_host_buffer(E: int, T: int, seed: int, device):
    from tianshou_b200.data import VectorReplayBuffer
    from tianshou_b200.synthetic import fill_vector_buffer
    buf = VectorReplayBuffer(E * T, E, device=device)
    fill_vector_buffer(buf, np.random.default_rng(seed), E, T, OBS, ACT)
    return buf


# ------------------------------------------------------------------------------- CPU baseline
def port_calibration() -> dict | None:
    """Build-box calibration of the port against the imported reference (tools/cpu_port_calibration.py)."""
    p = os.path.join(ROOT, "profiles", "cpu_port_calibration.json")
    if not os.path.exists(p):
        return None
    c = json.load(open(p))
    return {k: c[k] for k in ("port_over_reference", "reference_tps", "port_tps", "sample", "host_cores") if k in c}


def cpu_reference_run(E: int, T: int, steps: int, warmup: int, batch_size: int | None = None) -> dict:
    """numpy port of the reference's PPO update (oracle/oracle_np.py) on E x T transitions,
    same minibatch size / repeat / hyper-parameters; all host threads numpy's BLAS will use."""
    from oracle import oracle_np as onp
    from tianshou_b200.synthetic import synth_rollout
    try:  # the reference's `_gae` is compiled (numba): use the C restatement, not the Python loop
        from oracle import oracle_c
        oracle_c.lib()
        onp.gae = lambda v_s, v_s_, rew, end, gamma, lam: oracle_c.gae(v_s, v_s_, rew, end, gamma, lam)
    except OSError:
        pass
    rng = np.random.default_rng(0)
    cols: dict[str, list] = {k: [] for k in ("obs", "act", "rew", "terminated", "truncated", "obs_next")}
    for s in synth_rollout(rng, E, T, OBS, ACT):
        for k in cols:
            cols[k].append(s[k])
    # env-major flat order, like VectorReplayBuffer.sample(0)
    roll = {k: np.stack(v, axis=1).reshape(E * T, *v[0].shape[1:]) for k, v in cols.items()}
    N = E * T
    unf = np.zeros(N, dtype=bool)
    lastpos = np.arange(E) * T + T - 1
    unf[lastpos] = ~(roll["terminated"][lastpos] | roll["truncated"][lastpos])
    roll["unfinished"] = unf
    g = np.random.default_rng(1)
    def ortho(o, i, gain):
        a = g.standard_normal((o, i)); q, _ = np.linalg.qr(a.T if o < i else a); q = q.T if o < i else q
        return (gain * q[:o, :i]).astype(np.float32)
    p = {"a_w1": ortho(64, OBS, 2 ** .5), "a_b1": np.zeros(64, np.float32), "a_w2": ortho(64, 64, 2 ** .5),
         "a_b2": np.zeros(64, np.float32), "a_w3": 0.01 * ortho(ACT, 64, 2 ** .5), "a_b3": np.zeros(ACT, np.float32),
         "a_logstd": np.full((ACT, 1), -0.5, np.float32), "c_w1": ortho(64, OBS, 2 ** .5), "c_b1": np.zeros(64, np.float32),
         "c_w2": ortho(64, 64, 2 ** .5), "c_b2": np.zeros(64, np.float32), "c_w3": ortho(1, 64, 2 ** .5),
         "c_b3": np.zeros(1, np.float32)}
    m = {k: np.zeros_like(v) for k, v in p.items()}
    v = {k: np.zeros_like(x) for k, x in p.items()}
    hp = dict(eps_clip=0.2, dual_clip=None, vf_coef=0.25, ent_coef=0.0, max_grad_norm=0.5, adv_eps=1e-8, value_clip=True,
              advantage_normalization=False, lr=3e-4, beta1=0.9, beta2=0.999, adam_eps=1e-8, weight_decay=0.0)
    rms = onp.RunningMeanStd()
    step = 0

    def one_update() -> float:
        nonlocal step
        t0 = time.perf_counter()
        perms = [np.random.permutation(N) for _ in range(REPEAT)]
        res = onp.ppo_update(p, m, v, step, roll, perms, min(batch_size or BATCH_SIZE, N), REPEAT, hp, rms, 0.99, 0.95, True)
        step = res["step"]
        return time.perf_counter() - t0

    # "all the host threads it can use": the GEMMs are small (16384 x 64 x 64), so more BLAS threads is not
    # monotonically faster -- calibrate the thread count once (one update each) and time with the best one.
    ncpu = os.cpu_count() or 1
    cores, limiter = ncpu, None
    try:
        import threadpoolctl
        best = None
        for nthr in sorted({min(ncpu, c) for c in (4, 8, 16, 32, ncpu)}):
            with threadpoolctl.threadpool_limits(limits=nthr):
                dt = one_update()
            if best is None or dt < best[0]:
                best = (dt, nthr)
        cores = best[1]
        limiter = threadpoolctl.threadpool_limits(limits=cores)
    except ImportError:
        pass
    times = []
    for it in range(warmup + steps):
        dt = one_update()
        if it >= warmup:
            times.append(dt)
    if limiter is not None:
        limiter.restore_original_limits()
    mean_t = sum(times) / len(times)
    return {"value": N / mean_t, "unit": "transitions/s", "cores": int(cores), "kind": "port",
            "port_vs_imported_reference": port_calibration(),
            "sample": f"{E} envs x {T} steps = {N} transitions, minibatch {min(batch_size or BATCH_SIZE, N)}, repeat {REPEAT}, "
                      f"{len(times)} timed update() calls of the numpy port (oracle/oracle_np.py), "
                      f"{cores} BLAS threads (best of a calibration sweep over 4..{ncpu})",
            "ms_per_step": mean_t * 1e3}


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    E = int(os.environ.get("TS_BENCH_CPU_ENVS", "1024"))      # 1/4 of configs[1]: 8 minibatches of 16384 per pass
    res = cpu_reference_run(E, cfg["T"], args.steps, max(1, min(args.warmup, 1)))
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": "transitions/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus, args.config, args.scaling) | {"cpu_sample": res["sample"]},
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "port_vs_imported_reference")},
        "e2e": {"value": res["value"], "unit": "transitions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


CONFIGS = {   # BASELINE.json configs[1] and configs[4]
    "c2": {"E": E_FULL, "T": T_FULL, "bs": BATCH_SIZE, "name": "BASELINE configs[1]"},
    "c5": {"E": 8192, "T": 256, "bs": 8192 * 256 // 8, "name": "BASELINE configs[4]"},
}


def workload_config(n_gpus: int, config: str = "c2", scaling: str = "weak") -> dict:
    c = CONFIGS[config]
    per = "per GPU" if scaling == "weak" else f"in total, replicated on the {n_gpus} GPUs"
    return {"workload": f"PPO update(): synthetic HalfCheetah rollout {c['E']} envs x {c['T']} steps {per} "
                        f"(obs {OBS}, act {ACT}), MLP[64,64] tanh actor+critic, minibatch {c['bs']}"
                        f"{' per GPU' if scaling == 'weak' else ' split into ' + str(n_gpus) + ' contiguous slices'}, "
                        f"repeat {REPEAT}, recompute_advantage, value_clip, return_scaling ({c['name']})",
            "transitions": c["E"] * c["T"] * (n_gpus if scaling == "weak" else 1),
            "global_minibatch": c["bs"] * (n_gpus if scaling == "weak" else 1), "repeat": REPEAT,
            "parallelism": f"dp{n_gpus}", "scaling": scaling, "l2": "explicit 256 MiB L2 flush between timed update() calls",
            "minibatch_shuffle": "numpy (the default public API: the reference's np.random.permutation stream, bit-identical "
                                 "minibatch composition); the opt-in device-generated order is reported as *_device_order"}


def dump_outputs(out_dir: str, algo, actor, critic, batch) -> None:
    """What the caller of one headline step (``_preprocess_batch`` + ``_update_with_batch``) receives, as
    ``out_dir/<name>.npy``: the per-minibatch loss table, the running return statistics, the actor's and the critic's
    parameters, and the batch's per-transition ``v_s`` / ``returns`` / ``adv`` / ``logp_old``.  Rollouts longer than
    ``DUMP_ROWS`` contribute the rows listed in ``row_index`` (a fixed seeded sample) instead of every row."""
    import torch
    rms = algo.ret_rms
    out = {"loss_table": np.asarray(algo.last_loss_table, np.float64),
           "ret_rms": np.concatenate([np.asarray(x, np.float64).reshape(-1) for x in (rms.mean, rms.var, rms.count)])}
    for prefix, module in (("actor", actor), ("critic", critic)):
        for name, p in module.named_parameters():
            out[f"{prefix}.{name}"] = p.detach().float().cpu().numpy()
    n = batch.obs.shape[0]
    rows = None
    if n > DUMP_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
        out["row_index"] = rows.astype(np.float64)
    for key in ("v_s", "returns", "adv", "logp_old"):
        t = getattr(batch, key).detach()
        if rows is not None:
            t = t[torch.from_numpy(rows).to(t.device)]
        out[key] = t.float().cpu().numpy()
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte budget")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def positive_int(s: str) -> int:
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {v}")
    return v


# ------------------------------------------------------------------------------------ GPU arm
def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=5, help="timed update() calls per timed arm")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--envs", type=int, default=0, help="override the config's env count (diagnostics)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip config4 / ingest / off-policy extras")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline arm computed as DIR/<name>.npy (rank 0)")
    ap.add_argument("--profile-one-step", action="store_true",
                    help="after the warm-up run ONE end-to-end update() between cudaProfilerStart/Stop and exit (for "
                         "`ncu --profile-from-start off ...`: the launch list of exactly the timed step)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import hashlib

    import torch
    import torch.distributed as dist

    from tianshou_b200 import _cabi, ops
    from tianshou_b200._cabi import call, ptr, stream_ptr
    from tianshou_b200.data.batch import minibatch_bounds
    from tianshou_b200.synthetic import build_mujoco_ppo
    from tianshou_b200.utils import policy_within_training_step

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun)"
    _cabi.load_library()
    W = max(3, args.warmup)
    K = args.steps
    cfg = CONFIGS[args.config]
    E, T, BS = (args.envs or cfg["E"]), cfg["T"], cfg["bs"]
    N = E * T
    strong = args.scaling == "strong"
    part = "shared" if strong else "per_rank"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, iters: int) -> float:
        """sum of per-iteration device times (ms), L2 flushed before every iteration; max over ranks."""
        evs = []
        barrier()
        for _ in range(iters):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            evs.append((s, e))
        barrier()
        tot = sum(s.elapsed_time(e) for s, e in evs)
        if world > 1:
            t = torch.tensor([tot], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            tot = float(t.item())
        return tot

    def flat_hash(a) -> str:
        return hashlib.sha1(a._flat.flat.detach().cpu().numpy().tobytes()).hexdigest()[:16]

    def replicas_equal(a) -> bool:
        if world == 1:
            return True
        hs: list = [None] * world
        dist.all_gather_object(hs, flat_hash(a))
        return len(set(hs)) == 1

    # weak: every rank owns its own rollout; strong: ONE rollout (same seed) on every rank, same numpy stream
    buf = build_host_buffer(E, T, seed=0 if strong else rank, device=dev)
    np.random.seed(1000 if strong else 1000 + rank)
    algo, actor, critic = build_mujoco_ppo(OBS, ACT, dev, minibatch_shuffle="numpy", rollout_partition=part)         # default API
    algo_dv, _, _ = build_mujoco_ppo(OBS, ACT, dev, minibatch_shuffle="device", rollout_partition=part)

    with policy_within_training_step(algo.policy), policy_within_training_step(algo_dv.policy):
        dev_batch, dev_idx = algo._sample(buf, 0)

        def device_step(a=algo):
            with a._minibatch_order_job(buf, REPEAT):       # what update() does first: the minibatch-order draws start in the background
                b = a._preprocess_batch(dev_batch, buf, dev_idx)
                a._update_with_batch(b, BS, REPEAT)

        def e2e_step(a=algo):
            a.update(buffer=buf, batch_size=BS, repeat=REPEAT)

        if args.profile_one_step:
            for _ in range(W):
                e2e_step()
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
            e2e_step()
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
            print(json.dumps({"profiled": "one e2e update()", "config": workload_config(world, args.config, args.scaling)}))
            return

        # ---- headline: the DEFAULT public API (reference-exact minibatch order) ------------------------------
        for _ in range(W):
            device_step()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        _cabi.reset_launch_count()
        ms_dev = timed(device_step, K)
        launches = _cabi.launch_count()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, algo, actor, critic, dev_batch)
        for _ in range(W):
            e2e_step()
        ms_e2e = timed(e2e_step, K)
        clocks = sampler.stop() if rank == 0 else {}
        # ---- opt-in device-generated minibatch order (same kernels, no host permutation at all) --------------
        n_dv = max(1, min(K, 3))
        for _ in range(2):
            device_step(algo_dv)
        ms_dev_dv = timed(lambda: device_step(algo_dv), n_dv)
        e2e_step(algo_dv)
        ms_e2e_dv = timed(lambda: e2e_step(algo_dv), n_dv)
        main_replicas_equal = replicas_equal(algo) and replicas_equal(algo_dv)

        # ---- multi-GPU self-check, outside the timed region: N ranks (shared rollout, minibatch split N ways) vs ONE rank
        # on the same rollout / weights / permutation stream
        mg_check = None
        if world > 1:
            Ev, Tv, bsv, repv = 512, 128, 4096, 2
            vbuf = build_host_buffer(Ev, Tv, seed=4321, device=dev)
            a_n, _, _ = build_mujoco_ppo(OBS, ACT, dev, minibatch_shuffle="numpy", rollout_partition="shared")
            a_1, _, _ = build_mujoco_ppo(OBS, ACT, dev, minibatch_shuffle="numpy", data_parallel=False)
            tabs = []
            for a in (a_n, a_1):
                np_state = np.random.get_state()
                np.random.seed(99)
                with policy_within_training_step(a.policy):
                    a.update(buffer=vbuf, batch_size=bsv, repeat=repv)
                np.random.set_state(np_state)
                tabs.append(a.last_loss_table[:, :4].copy())
            loss_err = float(np.abs(tabs[0] - tabs[1]).max() / max(1e-30, np.abs(tabs[1]).max()))
            pn, p1 = a_n._flat.flat.detach().cpu().numpy(), a_1._flat.flat.detach().cpu().numpy()
            par_err = float(np.abs(pn - p1).max() / max(1e-30, np.abs(p1).max()))
            errs = torch.tensor([loss_err, par_err], dtype=torch.float64, device=dev)
            dist.all_reduce(errs, op=dist.ReduceOp.MAX)
            mg_check = {"replicas_equal": bool(replicas_equal(a_n) and main_replicas_equal),
                        "loss_rel_err": float(errs[0].item()), "param_rel_err": float(errs[1].item()),
                        "fused_peer_path": a_n._scratch.get("peer_exchange") is not None,
                        "what": f"{world} ranks (one shared rollout {Ev}x{Tv}, minibatch {bsv} split into {world} slices, same "
                                f"np.random stream) vs a single-rank update() of the same rollout on every rank: max |loss table "
                                f"difference| / max |loss|, max |parameter difference| / max |parameter| after {repv * (Ev * Tv // bsv)} "
                                "optimiser steps; replicas_equal = sha1 of the flat parameters identical on all ranks (this check "
                                "and the timed runs)"}

        # ---- BASELINE configs[4] (8192 x 256, minibatch N/8) strong-scaled over the N GPUs -------------------
        config4 = None
        if not args.no_extras and args.config == "c2":
            c5 = CONFIGS["c5"]
            if c5["bs"] % world == 0:
                buf5 = build_host_buffer(c5["E"], c5["T"], seed=5, device=dev)
                a5, _, _ = build_mujoco_ppo(OBS, ACT, dev, minibatch_shuffle="numpy", rollout_partition="shared")
                np_state = np.random.get_state()
                np.random.seed(55)
                with policy_within_training_step(a5.policy):
                    step5 = lambda: a5.update(buffer=buf5, batch_size=c5["bs"], repeat=REPEAT)   # noqa: E731
                    step5()
                    ms5 = timed(step5, 2)
                np.random.set_state(np_state)
                n5 = c5["E"] * c5["T"]
                a5d, _, _ = build_mujoco_ppo(OBS, ACT, dev, minibatch_shuffle="device", rollout_partition="shared")
                with policy_within_training_step(a5d.policy):
                    step5d = lambda: a5d.update(buffer=buf5, batch_size=c5["bs"], repeat=REPEAT)   # noqa: E731
                    step5d()
                    ms5d = timed(step5d, 2)
                del a5d
                config4 = {"value": n5 * 2 / (ms5 / 1e3), "unit": "transitions/s", "ms_per_step": ms5 / 2, "scaling": "strong",
                           "device_order": {"value": n5 * 2 / (ms5d / 1e3), "ms_per_step": ms5d / 2,
                                            "note": "same update() with the opt-in device-generated minibatch order: at 2 M transitions "
                                                    "the reference-exact order is bounded by the sequential MT19937 walk on the host "
                                                    "(~1.6 ms per 2 M-entry permutation), not by the GPUs"},
                           "n_gpus": world, "config": workload_config(world, "c5", "strong"), "steps": 2, "warmup": 1,
                           "timing": "end to end through update(): host rollout upload + D2H of the loss table inside",
                           "replicas_equal": replicas_equal(a5)}
                del buf5, a5

        # ---- rollout ingestion (SURVEY 8(f) rank 1): add() with the asynchronous device mirror, then an update()
        # that finds the rollout already on the device (no bulk upload in its timed region)
        ingest = None
        if world == 1 and not args.no_extras:
            from tianshou_b200.data import Batch, VectorReplayBuffer
            from tianshou_b200.synthetic import synth_rollout
            steps_host = [Batch(**s_) for s_ in synth_rollout(np.random.default_rng(7), E, T, OBS, ACT)]
            ids = np.arange(E)
            ingest = {}
            for mirror in (False, True):
                mb = VectorReplayBuffer(E * T, E, device=dev, device_mirror=mirror)
                mb.add(steps_host[0], buffer_ids=ids)           # allocation + (mirror) first bulk sync, untimed
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for s_ in steps_host[1:]:
                    mb.add(s_, buffer_ids=ids)
                t1 = time.perf_counter()
                torch.cuda.synchronize()
                t2 = time.perf_counter()
                ingest["mirror" if mirror else "host_only"] = {
                    "add_ms_per_call": 1e3 * (t1 - t0) / (T - 1), "transitions_per_s": E * (T - 1) / (t1 - t0),
                    "drain_ms_after_last_add": 1e3 * (t2 - t1)}
            from tianshou_b200.data import Batch as _B
            obs_host = steps_host[0].obs
            infer = {}
            for fused_on in (False, True):
                algo.policy.use_fused_inference = fused_on
                with torch.no_grad():
                    for _ in range(5):
                        algo.policy(_B(obs=obs_host, info=_B())).act.cpu()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(50):
                        algo.policy(_B(obs=obs_host, info=_B())).act.cpu()
                    infer["fused_kernel" if fused_on else "torch_modules"] = 1e6 * (time.perf_counter() - t0) / 50
            algo.policy.use_fused_inference = True
            ingest["policy_forward_us_per_call"] = infer | {"rows": int(E)}

            def e2e_mirrored_step():
                algo.update(buffer=mb, batch_size=BS, repeat=REPEAT)
            e2e_mirrored_step()
            ms_mir = timed(e2e_mirrored_step, K)
            ingest["update_from_mirror"] = {"value": N * K / (ms_mir / 1e3), "unit": "transitions/s", "ms_per_step": ms_mir / K,
                                            "note": "public update() on a buffer whose add() calls mirrored every row to the device "
                                                    "asynchronously during collection: no bulk H2D left in the update"}

    # ---- roofline of the dominant kernel: events around isolated launches on its stream -------
    hp = algo._ppo_hparams()
    f = algo._flat
    b = dev_batch
    perm = torch.randperm(N, device=dev).to(torch.int32)
    rows = min(BS, N)
    saved = [t.clone() for t in (f.flat, f.exp_avg, f.exp_avg_sq, f.step)]
    bounds = minibatch_bounds(N, BS, merge_last=True)
    epoch_stats = torch.zeros((len(bounds), 8), dtype=torch.float32, device=dev)
    epoch_events = []
    for i in range(10):     # the single-GPU product path: ONE persistent launch per pass over the rollout (all optimiser steps)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        algo._device_passes(b, perm, bounds, hp, epoch_stats, 1, False)
        e.record()
        if i >= 3:
            epoch_events.append((s, e))
    torch.cuda.synchronize()
    for dst, src in zip((f.flat, f.exp_avg, f.exp_avg_sq, f.step), saved):
        dst.copy_(src)
    epoch_ms = sum(s.elapsed_time(e) for s, e in epoch_events) / len(epoch_events)
    fwd_events = []
    for i in range(8):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        ops.critic_forward(f.flat, algo._desc, b.obs, b.obs_next, out=b.v_s, out2=algo._buf("v_next", N, torch.float32))
        e.record()
        if i >= 2:
            fwd_events.append((s, e))
    torch.cuda.synchronize()
    fwd_ms = sum(s.elapsed_time(e) for s, e in fwd_events) / len(fwd_events)
    gae_events = []
    for i in range(25):     # GAE scan alone (HBM-bound kernel), L2 flushed
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        ops.gae(b.v_s, algo._buf("v_next", N, torch.float32), b.rew, b.terminated, b.truncated, b.get("_unfinished"),
                gamma=0.99, gae_lambda=0.95, out=(b.adv, b.returns), workspace=algo._gae_workspace(N))
        e.record()
        if i >= 5:
            gae_events.append((s, e))
    torch.cuda.synchronize()
    gae_ms = sum(s.elapsed_time(e) for s, e in gae_events) / len(gae_events)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_src = load_peaks()
    total_transitions = N * (1 if strong else world)
    value = total_transitions * K / (ms_dev / 1e3)
    e2e_value = total_transitions * K / (ms_e2e / 1e3)
    meta_bytes = buf._extend_offset.nbytes + buf.last_index.nbytes + buf._sizes.nbytes
    h2d = sum(np.asarray(buf._meta[k]).nbytes for k in ("obs", "obs_next", "act", "rew", "terminated", "truncated", "done")) + meta_bytes
    h2d += REPEAT * N * 4                       # the host-drawn permutations (int32) of the default minibatch order
    n_mb = len(bounds)
    d2h = REPEAT * n_mb * 8 * 4 + 3 * 8
    grad_flops = FLOP_TRAIN_PER_ROW * N            # one pass of the epoch kernel touches every transition once
    grad_tflops = grad_flops / (epoch_ms * 1e-3) / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("ppo_epoch_kernel_dram_bytes_per_launch")
    gae_bytes = 27 * N
    line = {
        "metric": METRIC, "value": value, "unit": "transitions/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32 (MLP fwd/bwd, Adam), f64 (GAE scan, running return statistics)", "data": "synthetic",
        "config": workload_config(world, args.config, args.scaling),
        "e2e": {"value": e2e_value, "unit": "transitions/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": ms_e2e / K},
        "value_device_order": {"value": total_transitions * n_dv / (ms_dev_dv / 1e3), "unit": "transitions/s", "ms_per_step": ms_dev_dv / n_dv},
        "e2e_device_order": {"value": total_transitions * n_dv / (ms_e2e_dv / 1e3), "unit": "transitions/s", "ms_per_step": ms_e2e_dv / n_dv,
                             "note": "opt-in minibatch_shuffle='device' (ts_make_permutation): same kernels, the minibatch order is a "
                                     "keyed bijection generated on the GPU instead of the reference's np.random.permutation stream"},
        "default_over_device_order": {"value": (ms_dev_dv / n_dv) / (ms_dev / K), "e2e": (ms_e2e_dv / n_dv) / (ms_e2e / K)},
        "gpu_launches": int(launches),
        "multi_gpu_check": mg_check,
        "config4": config4,
        "ingest": ingest,
        "roofline": {"kernel": "ppo_tc_kernel<EPOCH> (persistent: every optimiser step of one pass = minibatch fwd/bwd + "
                               "gradient fold + clip + Adam; tcgen05 bf16x3 = fp32-faithful)", "bound": "tensor",
                     "achieved": grad_tflops, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                     "frac": grad_tflops / peaks["bf16_tflops"], "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_flops_per_launch": grad_flops, "launch_ms": epoch_ms, "rows_per_launch": N,
                     "optimiser_steps_per_launch": len(bounds), "us_per_optimiser_step": 1e3 * epoch_ms / len(bounds),
                     "note": "latency-bound chain of dependent MMA stages per 128-row tile on a 17-64-64-{1,6} MLP; forward and input-"
                             "gradient GEMMs use 6 bf16 MMAs per algorithmic one (fp32-faithful), weight-gradient GEMMs 3"},
        "roofline_gae": {"kernel": "gae_scan_kernel", "bound": "hbm", "achieved": gae_bytes / (gae_ms * 1e-3) / 1e9,
                         "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gae_bytes / (gae_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                         "algorithmic_bytes_per_launch": gae_bytes, "launch_ms": gae_ms, "peak_source": peak_src},
        "kernel_ms": {"ppo_epoch(all optimiser steps of one pass)": epoch_ms, "critic_forward(v_s,v_s_)": fwd_ms, "gae_scan": gae_ms},
        "flops_per_transition": FLOP_PER_TRANSITION,
        "update_tflops": FLOP_PER_TRANSITION * total_transitions * K / (ms_dev / 1e3) / 1e12,
        "clocks": clocks,
    }
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_run(int(os.environ.get("TS_BENCH_CPU_ENVS_INLINE", "256")), T, 3, 1, batch_size=BS)
        line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "port_vs_imported_reference")}
    if world == 1 and not args.no_extras:
        try:
            line["offpolicy"] = offpolicy_extras(dev)
        except Exception as ex:  # noqa: BLE001 - extras must never take the headline down
            line["offpolicy"] = {"error": repr(ex)}
        try:        # context only (SURVEY 2.3): the reference's own style of update with stock PyTorch on the same GPU
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import torch_eager_context
            line["context_torch_eager_gpu"] = torch_eager_context.run(E=E, T=T, bs=BS, repeat=REPEAT, steps=1, device=str(dev))
        except Exception as ex:  # noqa: BLE001
            line["context_torch_eager_gpu"] = {"error": repr(ex)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def offpolicy_extras(dev) -> dict:
    """BASELINE configs[2] / configs[3] shaped ``update()`` calls (SURVEY 8(f) ranks 2-3): updates/s of the device path through
    the public API next to the torch-CPU restatement (oracle/oracle_offpolicy.py) on the same shapes.  Buffer sizes are reduced
    from the 1 M / 4 M transitions BASELINE names (stated in ``workload``): the update cost does not depend on the buffer size,
    only the host memory of the synthetic fill does."""
    import copy

    import torch

    from oracle import oracle_offpolicy as oo
    from tianshou_b200.algorithm import AdamOptimizerFactory
    from tianshou_b200.algorithm.modelfree.dqn import DQN, DiscreteQLearningPolicy
    from tianshou_b200.algorithm.modelfree.sac import SAC, SACPolicy
    from tianshou_b200.data import Batch, PrioritizedVectorReplayBuffer, VectorReplayBuffer
    from tianshou_b200.env.atari import DQNet, ScaledObsInputActionReprNet
    from tianshou_b200.synthetic import BoxSpace
    from tianshou_b200.utils import policy_within_training_step
    from tianshou_b200.utils.net.common import Net
    from tianshou_b200.utils.net.continuous import ContinuousActorProbabilistic, ContinuousCritic

    out: dict = {}
    rng = np.random.default_rng(0)
    # batch-256 MLPs / batch-32 convolutions do not scale past a few cores: give the CPU port its best case, not every core
    cpu_threads = min(8, os.cpu_count() or 1)
    torch.set_num_threads(cpu_threads)

    def time_updates(fn, warm: int, iters: int) -> float:
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / iters

    # ---- SAC, Humanoid-shaped (obs 376, act 17, MLP[256,256], batch 256; examples/mujoco/mujoco_sac.py:29-44) ------------
    O, A, H, B = 376, 17, (256, 256), 256
    E, steps = 64, 1024
    torch.manual_seed(0)
    actor = ContinuousActorProbabilistic(preprocess_net=Net(state_shape=(O,), hidden_sizes=H), action_shape=(A,), unbounded=True,
                                         conditioned_sigma=True).to(dev)
    c1 = ContinuousCritic(preprocess_net=Net(state_shape=(O,), action_shape=(A,), hidden_sizes=H, concat=True)).to(dev)
    c2 = ContinuousCritic(preprocess_net=Net(state_shape=(O,), action_shape=(A,), hidden_sizes=H, concat=True)).to(dev)
    cpu_nets = oo.SacNets(O, A, H)
    with torch.no_grad():
        for dst, src in zip(cpu_nets.actor_params(), actor.parameters(), strict=True):
            dst.copy_(src.cpu())
        for k, c in enumerate((c1, c2)):
            for dst, src in zip(cpu_nets.c[k].parameters(), c.parameters(), strict=True):
                dst.copy_(src.cpu())
    cpu_nets.c_old = [copy.deepcopy(c) for c in cpu_nets.c]
    graph_nets = copy.deepcopy((actor, c1, c2))

    def make_sac(a, q1, q2, **kw):
        return SAC(policy=SACPolicy(actor=a, action_space=BoxSpace(A)), policy_optim=AdamOptimizerFactory(lr=1e-3), critic=q1,
                   critic_optim=AdamOptimizerFactory(lr=1e-3), critic2=q2, critic2_optim=AdamOptimizerFactory(lr=1e-3), tau=0.005,
                   gamma=0.99, alpha=0.2, n_step_return_horizon=1, **kw)
    algo = make_sac(actor, c1, c2)
    buf = VectorReplayBuffer(E * steps, E, device=dev, device_mirror=True)
    obs = rng.standard_normal((E, O)).astype(np.float32)
    for _ in range(steps):
        nxt = rng.standard_normal((E, O)).astype(np.float32)
        buf.add(Batch(obs=obs, act=np.tanh(rng.standard_normal((E, A))).astype(np.float32), rew=rng.standard_normal(E),
                      terminated=rng.random(E) < 1e-3, truncated=np.zeros(E, bool), obs_next=nxt), buffer_ids=np.arange(E))
        obs = nxt
    with policy_within_training_step(algo.policy):
        dt = time_updates(lambda: algo.update(buffer=buf, sample_size=B), 5, 50)
    algo_g = make_sac(*graph_nets, cuda_graph=True)          # same update, device work replayed from one CUDA graph
    with policy_within_training_step(algo_g.policy):
        dt_g = time_updates(lambda: algo_g.update(buffer=buf, sample_size=B), 5, 200)
    graph_ok = algo_g._graph.get("graph") is not None
    host = dict(obs=np.asarray(buf.obs), act=np.asarray(buf.act), rew=np.asarray(buf.rew), done=np.asarray(buf.done),
                terminated=np.asarray(buf.terminated), obs_next=np.asarray(buf.obs_next), offset=np.asarray(buf._extend_offset),
                last_index=np.asarray(buf.last_index), lengths=np.asarray(buf._sizes))
    opts = [torch.optim.Adam(cpu_nets.actor_params(), lr=1e-3)] + [torch.optim.Adam(cpu_nets.c[k].parameters(), lr=1e-3) for k in range(2)]

    def cpu_sac():
        idx = rng.integers(0, E * steps, B)
        oo.sac_update(cpu_nets, opts, host, idx, torch.randn(B, A), torch.randn(B, A), 0.99, 1, 0.2, 0.005)
    cpu_sac()
    t0 = time.perf_counter()
    for _ in range(20):
        cpu_sac()
    dt_cpu = (time.perf_counter() - t0) / 20
    out["sac"] = {"updates_per_s": 1.0 / dt, "transitions_per_s": B / dt, "ms_per_update": 1e3 * dt,
                  "cuda_graph": {"updates_per_s": 1.0 / dt_g, "ms_per_update": 1e3 * dt_g, "replaying": bool(graph_ok),
                                 "note": "SAC(cuda_graph=True): index draw + noise on the host/eager side, everything else one graph replay"},
                  "cpu_port": {"updates_per_s": 1.0 / dt_cpu, "ms_per_update": 1e3 * dt_cpu, "kind": "port (torch CPU, oracle/oracle_offpolicy.py)",
                               "threads": torch.get_num_threads()},
                  "workload": f"SAC.update(sample_size={B}) obs {O} act {A} MLP{list(H)} actor + 2 critics + 2 lagged critics, "
                              f"VectorReplayBuffer {E * steps} transitions with device mirror (BASELINE configs[3] names 4 M), 1 GPU"}
    del buf, algo, algo_g

    # ---- DQN, Atari-shaped (84x84x4 uint8, NatureCNN, PER, 3-step, batch 32; examples/atari/atari_dqn.py:34-49) ----------
    Hh, Ww, NA, B = 84, 84, 6, 32
    E, steps = 16, 2048
    torch.manual_seed(0)
    net = ScaledObsInputActionReprNet(DQNet(4, Hh, Ww, NA)).to(dev)
    cpu_net = oo.nature_cnn(4, Hh, Ww, NA)
    with torch.no_grad():
        for dst, src in zip(cpu_net.parameters(), net.parameters(), strict=True):
            dst.copy_(src.cpu())
    cpu_old = copy.deepcopy(cpu_net)
    dqn = DQN(policy=DiscreteQLearningPolicy(model=net, action_space=type("D", (), {"n": NA, "shape": ()})()), optim=AdamOptimizerFactory(lr=1e-4),
              gamma=0.99, n_step_return_horizon=3, target_update_freq=500, is_double=True)
    buf = PrioritizedVectorReplayBuffer(E * steps, E, alpha=0.6, beta=0.4, stack_num=4, ignore_obs_next=True, save_only_last_obs=True,
                                        device=dev, device_mirror=True)
    for _ in range(steps):
        fr = rng.integers(0, 256, (E, 1, Hh, Ww), dtype=np.uint8)
        st = np.broadcast_to(fr, (E, 4, Hh, Ww))
        buf.add(Batch(obs=st, act=rng.integers(0, NA, E), rew=rng.standard_normal(E), terminated=rng.random(E) < 2e-3,
                      truncated=np.zeros(E, bool), obs_next=st), buffer_ids=np.arange(E))
    with policy_within_training_step(dqn.policy):
        dt = time_updates(lambda: dqn.update(buffer=buf, sample_size=B), 5, 50)
    host = dict(obs=np.asarray(buf.obs), act=np.asarray(buf.act).astype(np.int64), rew=np.asarray(buf.rew), done=np.asarray(buf.done),
                terminated=np.asarray(buf.terminated), offset=np.asarray(buf._extend_offset), last_index=np.asarray(buf.last_index),
                lengths=np.asarray(buf._sizes))
    opt = torch.optim.Adam(cpu_net.parameters(), lr=1e-4)

    def cpu_dqn():
        idx = rng.integers(0, E * steps, B)
        oo.dqn_update(cpu_net, cpu_old, opt, host, idx, np.ones(B, np.float32), 0.99, 3, True, None)
    cpu_dqn()
    t0 = time.perf_counter()
    for _ in range(10):
        cpu_dqn()
    dt_cpu = (time.perf_counter() - t0) / 10
    out["dqn"] = {"updates_per_s": 1.0 / dt, "transitions_per_s": B / dt, "ms_per_update": 1e3 * dt,
                  "cpu_port": {"updates_per_s": 1.0 / dt_cpu, "ms_per_update": 1e3 * dt_cpu, "kind": "port (torch CPU, oracle/oracle_offpolicy.py)",
                               "threads": torch.get_num_threads()},
                  "workload": f"DQN.update(sample_size={B}): NatureCNN on 84x84x4 uint8 frame stacks gathered from single-frame storage, "
                              f"double DQN, 3-step return, PrioritizedVectorReplayBuffer {E * steps} frames with device mirror "
                              "(BASELINE configs[2] names 1 M), 1 GPU"}
    return out


if __name__ == "__main__":
    main()
