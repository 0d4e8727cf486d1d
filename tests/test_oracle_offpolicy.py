"""Pin the torch-CPU restatement of the off-policy update bodies (oracle/oracle_offpolicy.py) to outputs of the imported
reference (tests/golden/sac_ref.npz, dqn_ref*.npz).  CPU only."""
import copy

import numpy as np
import pytest
import torch

from oracle import oracle_offpolicy as oo
from ts_testutil import load_dqn_golden, load_golden


def _load(params, g, prefix):
    with torch.no_grad():
        for i, p in enumerate(params):
            p.copy_(torch.as_tensor(g[f"{prefix}{i}"]).reshape(p.shape))


def _close(params, g, prefix, lr, what):
    for i, p in enumerate(params):
        np.testing.assert_allclose(p.detach().numpy(), g[f"{prefix}{i}"], rtol=1e-3, atol=0.1 * lr, err_msg=f"{what} {prefix}{i}")


def test_sac_oracle_matches_reference_run():
    g = load_golden("sac_ref.npz")
    O, A, H = int(g["cfg_obs"]), int(g["cfg_act"]), tuple(int(x) for x in g["cfg_hidden"])
    lr, E, cap = float(g["cfg_lr"]), int(g["cfg_E"]), int(g["cfg_cap"])
    nets = oo.SacNets(O, A, H)
    _load(nets.actor_params(), g, "p0_actor_")
    for k in range(2):
        _load(list(nets.c[k].parameters()), g, f"p0_c{k + 1}_")
    nets.c_old = [copy.deepcopy(c) for c in nets.c]
    opts = [torch.optim.Adam(nets.actor_params(), lr=lr)] + [torch.optim.Adam(nets.c[k].parameters(), lr=lr) for k in range(2)]
    buf = dict(obs=g["buf_obs"], act=g["buf_act"], rew=g["buf_rew"], done=g["buf_done"], terminated=g["buf_terminated"],
               obs_next=g["buf_obs_next"], offset=np.arange(E + 1) * cap, last_index=g["meta_last_index"], lengths=g["meta_lengths"])
    B = int(g["cfg_bs"])
    for u in range(int(g["cfg_updates"])):
        torch.manual_seed(100 + u)
        n1 = torch.normal(torch.zeros(B, A), torch.ones(B, A))
        n2 = torch.normal(torch.zeros(B, A), torch.ones(B, A))
        o = f"u{u}_"
        res = oo.sac_update(nets, opts, buf, g[o + "indices"], n1, n2, float(g["cfg_gamma"]), int(g["cfg_n_step"]), float(g["cfg_alpha"]),
                            float(g["cfg_tau"]))
        np.testing.assert_allclose(res["returns"], g[o + "returns"].reshape(-1), rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose([res["actor_loss"], res["critic1_loss"], res["critic2_loss"]], g[o + "losses"], rtol=1e-5, atol=1e-6)
        _close(nets.actor_params(), g, o + "actor_", lr, "actor")
        for k in range(2):
            _close(list(nets.c[k].parameters()), g, o + f"c{k + 1}_", lr, "critic")
            _close(list(nets.c_old[k].parameters()), g, o + f"c{k + 1}old_", lr, "lagged critic")


@pytest.mark.parametrize("variant", ["", "_b"])
def test_dqn_oracle_matches_reference_run(variant):
    g = load_dqn_golden(variant)
    H, W, A, E, cap = (int(g["cfg_" + k]) for k in ("H", "W", "A", "E", "cap"))
    lr = float(g["cfg_lr"])
    net = oo.nature_cnn(4, H, W, A)
    _load(list(net.parameters()), g, "p0_q_")
    freq = int(g["cfg_target_freq"])
    net_old = copy.deepcopy(net)
    opt = torch.optim.Adam(net.parameters(), lr=lr)
    # storage replayed on the host exactly as the buffer lays it out: env e owns [e * cap, (e + 1) * cap), slot t % cap
    steps = int(g["cfg_steps"])
    frames = np.zeros((E * cap, H, W), np.uint8)
    act = np.zeros(E * cap, np.int64); rew = np.zeros(E * cap); done = np.zeros(E * cap, bool); term = np.zeros(E * cap, bool)
    for t in range(steps):
        slots = np.arange(E) * cap + t % cap
        frames[slots], act[slots], rew[slots] = g[f"roll{t}_obs"], g[f"roll{t}_act"], g[f"roll{t}_rew"]
        term[slots] = g[f"roll{t}_terminated"]
        done[slots] = g[f"roll{t}_terminated"] | g[f"roll{t}_truncated"]
    buf = dict(obs=frames, act=act, rew=rew, done=done, terminated=term, offset=np.arange(E + 1) * cap,
               last_index=np.arange(E) * cap + (steps - 1) % cap, lengths=np.full(E, min(steps, cap)))
    huber = float(g["cfg_huber"])
    n_up = int(g["cfg_updates"])
    for u in range(n_up):
        o = f"u{u}_"
        res = oo.dqn_update(net, net_old if freq > 0 else None, opt, buf, g[o + "indices"], g[o + "is_weight"], float(g["cfg_gamma"]),
                            int(g["cfg_n_step"]), bool(g["cfg_is_double"]), None if np.isnan(huber) else huber,
                            sync_target=freq > 0 and u % freq == 0)
        np.testing.assert_allclose(res["returns"], g[o + "returns"].reshape(-1), rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(res["td"], g[o + "td"], rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(res["loss"], float(g[o + "loss"]), rtol=1e-5, atol=1e-6)
    _close(list(net.parameters()), g, f"u{n_up - 1}_q_", lr, "q")
    if freq > 0:
        _close(list(net_old.parameters()), g, f"u{n_up - 1}_qold_", lr, "lagged q")
