"""IPPO (marlbase/ac/model.py PPONetwork, 249-352): the oracle restatement against recorded outputs of the reference classes (tests/golden/ref_ppo.npz),
and the B200 path (marl_ppo_update through ac.model.PPONetwork) against the oracle on random on-policy batches; driver test."""
import os
import types

import numpy as np
import pytest
import torch

from oracle import learner_ref as lr
from tests.helpers import load_case, net_layers, sample_index

N, D, A, T = 2, 15, 6, 25


def _close(a, b, rtol=1e-5, atol=1e-5):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert np.allclose(a, b, rtol=rtol, atol=atol), float(np.abs(a - b).max())


def _space(shape=None, n=None):
    return types.SimpleNamespace(shape=shape, n=n)


def _batch_arrays(rng, P, n_agents):
    obs = rng.integers(-1, 8, size=(P, n_agents, T + 1, D)).astype(np.float32)
    act = rng.integers(0, A, size=(P, n_agents, T)).astype(np.int32)
    rew = (rng.random((P, n_agents, T)) < 0.2).astype(np.float32) * rng.random((P, n_agents, T)).astype(np.float32)
    length = rng.integers(1, T + 1, size=P)
    done = np.zeros((P, T + 1), np.uint8); filled = np.zeros((P, T), np.uint8)
    for e in range(P):
        filled[e, : length[e]] = 1
        done[e, length[e]] = 1
    return dict(obs=obs, act=act, rew=rew, done=done, filled=filled)


def _oracle_batch(s):
    t = {k: torch.as_tensor(v) for k, v in s.items()}
    P, n_agents = t["obs"].shape[0], t["obs"].shape[1]
    return dict(obss=t["obs"].permute(2, 0, 1, 3).reshape(T + 1, P, n_agents * D).float(), actions=t["act"].permute(2, 0, 1).long(),
                rewards=t["rew"].permute(2, 0, 1).float(), dones=t["done"].permute(1, 0).float(), filled=t["filled"].permute(1, 0).float())


METRICS = ("loss", "actor_loss", "value_loss", "entropy")
LIVE = os.path.join(os.path.dirname(__file__), "golden", "ref_ppo.npz")
# the reference runs recorded by make_reference_cases: name -> (class, torch seed, batch seed, envs per batch, update steps, config, critic config)
LIVE_CASES = {
    "std_A2CNetwork": ("A2CNetwork", 9, 3, 10, (0, 2, 3), dict(standardise_returns=True, num_epochs=3, ppo_clip=0.2, target_update_interval_or_tau=2), {}),
    "std_PPONetwork": ("PPONetwork", 9, 3, 10, (0, 2, 3), dict(standardise_returns=True, num_epochs=3, ppo_clip=0.2, target_update_interval_or_tau=2), {}),
    "cent_A2CNetwork": ("A2CNetwork", 4, 5, 10, (0, 2, 3), dict(num_epochs=3, ppo_clip=0.2, target_update_interval_or_tau=2), dict(centralised=True)),
    "cent_PPONetwork": ("PPONetwork", 4, 5, 10, (0, 2, 3), dict(num_epochs=3, ppo_clip=0.2, target_update_interval_or_tau=2), dict(centralised=True)),
    "ppo_indep_noclip": ("PPONetwork", 5, 11, 12, (0, 2, 5), dict(grad_clip=False, num_epochs=4, ppo_clip=0.2, target_update_interval_or_tau=2), {}),
    "ppo_shared_clip": ("PPONetwork", 5, 11, 12, (0, 2, 5), dict(grad_clip=0.5, num_epochs=4, ppo_clip=0.2, target_update_interval_or_tau=2), dict(parameter_sharing=True)),
}


def _live_layout(case):
    """(n_nets, critic input width, sample positions of the actor, of the critic) of a recorded case"""
    crit = LIVE_CASES[case][6]
    n_nets = 1 if crit.get("parameter_sharing") else N
    c_in = N * D if crit.get("centralised") else D
    return n_nets, c_in, sample_index(net_layers(n_nets, D, A)), sample_index(net_layers(n_nets, c_in, 1))


def make_reference_cases():
    """Records tests/golden/ref_ppo.npz from the reference's A2CNetwork / PPONetwork: MARLBASE_SRC=<marlbase checkout> python -c 'import
    tests.test_ppo as t; t.make_reference_cases()'.  Per case: the metrics of each update, the return statistics, and the parameters before and after
    at the positions of _live_layout."""
    from collections import namedtuple

    from oracle import ref_shim

    ref = ref_shim.load()
    Batch = namedtuple("Batch", ["obss", "actions", "rewards", "dones", "filled", "action_masks"])
    out = {}
    for case, (cls, seed, bseed, P, steps, cfgkw, critkw) in LIVE_CASES.items():
        n_nets, c_in, ia, ic = _live_layout(case)
        kind = "networks" if n_nets == 1 else "independent"
        torch.manual_seed(seed)
        net = ref_shim.net_cfg(parameter_sharing=bool(critkw.get("parameter_sharing")))
        model = getattr(ref.ac_model, cls)([ref_shim.Space(shape=(D,))] * N, [ref_shim.Space(n=A)] * N, ref_shim.a2c_cfg(**cfgkw), net, ref_shim.net_cfg(**critkw), "cpu")
        sd = model.state_dict()
        out[f"{case}.critic_in"] = np.int64(sd[f"critic.{kind}.0.network.0.weight"].shape[1])
        out[f"{case}.actor0"] = lr.flat_from_state_dict(sd, f"actor.{kind}", n_nets).numpy()[ia]
        out[f"{case}.critic0"] = lr.flat_from_state_dict(sd, f"critic.{kind}", n_nets).numpy()[ic]
        out[f"{case}.target0"] = lr.flat_from_state_dict(sd, f"target_critic.{kind}", n_nets).numpy()[ic]
        rng = np.random.default_rng(bseed)
        metrics = []
        for step in steps:
            b = _oracle_batch(_batch_arrays(rng, P, N))
            want = model.update(Batch(b["obss"], b["actions"], b["rewards"], b["dones"].bool(), b["filled"], None), step)
            metrics.append([want[k] for k in METRICS])
        out[f"{case}.metrics"] = np.array(metrics, np.float64)
        if cfgkw.get("standardise_returns"):
            out.update({f"{case}.ret_mean": model.ret_ms.mean.numpy(), f"{case}.ret_var": model.ret_ms.var.numpy(), f"{case}.ret_count": np.float64(model.ret_ms.count)})
        sd = model.state_dict()
        out.update({f"{case}.actor": lr.flat_from_state_dict(sd, f"actor.{kind}", n_nets).numpy()[ia],
                    f"{case}.critic": lr.flat_from_state_dict(sd, f"critic.{kind}", n_nets).numpy()[ic],
                    f"{case}.target": lr.flat_from_state_dict(sd, f"target_critic.{kind}", n_nets).numpy()[ic]})
    np.savez_compressed(LIVE, **out)


def _live_state(case, g, **kw):
    """The oracle's state from the reference's initialisation (torch seed of the case; actor drawn before critic, the target critic is a copy)"""
    n_nets, c_in, ia, ic = _live_layout(case)
    assert int(g["critic_in"]) == c_in
    torch.manual_seed(LIVE_CASES[case][1])
    actor, critic = lr.init_flat(n_nets, D, A), lr.init_flat(n_nets, c_in, 1)
    for mine, key, idx in ((actor, "actor0", ia), (critic, "critic0", ic), (critic, "target0", ic)):
        assert np.abs(mine.numpy()[idx] - g[key]).max() < 1e-6, f"initialisation differs from the reference's ({key})"
    nets = [0] * N if n_nets == 1 else list(range(N))
    return lr.A2CState(actor, critic, critic.clone(), nets, nets, D, A, **kw), ia, ic


def _run_live_case(case, st, update):
    g = load_case(LIVE, case)
    rng = np.random.default_rng(LIVE_CASES[case][2])
    for step, want in zip(LIVE_CASES[case][4], g["metrics"]):
        got = update(st, _oracle_batch(_batch_arrays(rng, LIVE_CASES[case][3], N)), step)
        _close([got[k] for k in METRICS], want)
    return g


@pytest.mark.parametrize("cls", ["A2CNetwork", "PPONetwork"])
def test_oracle_standardise_returns_matches_live_reference(cls):
    """cfg.standardise_returns=True: RunningMeanStd over the n-step returns (ac/model.py:195-204, 272-281) -- oracle vs what the reference's classes
    computed (tests/golden/ref_ppo.npz)"""
    case = f"std_{cls}"
    st, ia, _ = _live_state(case, load_case(LIVE, case), ret_ms=lr.RunningMeanStdRef((N,)))
    hp = lr.A2CHP(target_update_interval_or_tau=2)
    g = _run_live_case(case, st, lambda st, b, step: lr.ppo_update(st, b, hp, step, 3, 0.2) if cls == "PPONetwork" else lr.a2c_update(st, b, hp, step))
    _close(st.ret_ms.mean.numpy(), g["ret_mean"]); _close(st.ret_ms.var.numpy(), g["ret_var"])
    assert abs(st.ret_ms.count - float(g["ret_count"])) < 1e-9
    d = np.abs(st.actor.numpy()[ia] - g["actor"])
    assert np.quantile(d, 0.999) < 1e-5


@pytest.mark.parametrize("cls", ["A2CNetwork", "PPONetwork"])
def test_oracle_centralised_critic_matches_live_reference(cls):
    """critic.centralised=True (MAA2C / MAPPO, ac/model.py:62-65,156-157): oracle vs what the reference's classes computed (tests/golden/ref_ppo.npz)"""
    case = f"cent_{cls}"
    st, _, ic = _live_state(case, load_case(LIVE, case), centralised=True)
    hp = lr.A2CHP(target_update_interval_or_tau=2)
    g = _run_live_case(case, st, lambda st, b, step: lr.ppo_update(st, b, hp, step, 3, 0.2) if cls == "PPONetwork" else lr.a2c_update(st, b, hp, step))
    d = np.abs(st.critic.numpy()[ic] - g["critic"])
    assert np.quantile(d, 0.999) < 1e-5


@pytest.mark.parametrize("sharing,clip", [(False, False), (True, 0.5)])
def test_oracle_ppo_matches_live_reference(sharing, clip):
    """three PPO updates (4 epochs each) of oracle.learner_ref.ppo_update vs what the reference's PPONetwork computed from the same weights and
    batches (tests/golden/ref_ppo.npz)"""
    case = "ppo_shared_clip" if sharing else "ppo_indep_noclip"
    assert LIVE_CASES[case][5]["grad_clip"] == clip
    st, ia, ic = _live_state(case, load_case(LIVE, case))
    hp = lr.A2CHP(grad_clip=float(clip or 0.0), target_update_interval_or_tau=2)
    g = _run_live_case(case, st, lambda st, b, step: lr.ppo_update(st, b, hp, step, 4, 0.2))
    for mine, key, idx in ((st.actor, "actor", ia), (st.critic, "critic", ic), (st.target, "target", ic)):
        d = np.abs(mine.numpy()[idx] - g[key])
        assert np.quantile(d, 0.999) < 1e-5, (key, d.max())


def test_oracle_ppo_first_epoch_is_a2c_with_unit_ratio():
    """epoch 0: ratio == 1 exactly, inside the clip range -> the surrogate's gradient is the policy gradient of A2C"""
    rng = np.random.default_rng(2)
    theta_a, theta_c = lr.init_flat(N, D, A), lr.init_flat(N, D, 1)
    b = _oracle_batch(_batch_arrays(rng, 8, N))
    st1 = lr.A2CState(theta_a.clone(), theta_c.clone(), theta_c.clone(), [0, 1], [0, 1], D, A)
    st2 = lr.A2CState(theta_a.clone(), theta_c.clone(), theta_c.clone(), [0, 1], [0, 1], D, A)
    g_ppo = lr.ppo_update(st1, b, lr.A2CHP(), 0, 1, 0.2)["grad"]
    g_a2c = lr.a2c_update(st2, b, lr.A2CHP(), 0)["grad"]
    _close(g_ppo["actor"].numpy(), g_a2c["actor"].numpy()); _close(g_ppo["critic"].numpy(), g_a2c["critic"].numpy())


def _model(sharing, hp, P, n_agents, num_epochs, ppo_clip, standardise=False, cls="PPONetwork", centralised=False):
    from codebase_b200.ac import model as M

    cfg = types.SimpleNamespace(optimizer="Adam", lr=hp.lr, gamma=hp.gamma, grad_clip=hp.grad_clip, n_steps=hp.n_steps, entropy_coef=hp.entropy_coef,
                                value_loss_coef=hp.value_loss_coef, target_update_interval_or_tau=hp.target_update_interval_or_tau, standardise_returns=standardise,
                                num_epochs=num_epochs, ppo_clip=ppo_clip)
    net = types.SimpleNamespace(layers=[128, 128], parameter_sharing=sharing, use_rnn=False, use_orthogonal_init=True, centralised=False)
    cnet = types.SimpleNamespace(layers=[128, 128], parameter_sharing=sharing, use_rnn=False, use_orthogonal_init=True, centralised=centralised)
    return getattr(M, cls)([_space(shape=(D,))] * n_agents, [_space(n=A)] * n_agents, cfg, net, cnet, "cuda", max_envs=P, max_episode_length=T)


@pytest.mark.gpu
@pytest.mark.parametrize("sharing,P,n_agents,clip,epochs,lr_", [(False, 64, 2, 0.0, 4, 3e-4), (True, 500, 2, 0.5, 4, 3e-4), ([0, 1, 0], 96, 3, 0.0, 2, 3e-4),
                                                               (False, 128, 2, 0.5, 6, 3e-3)])   # the last: a learning rate that drives ratios out of the clip range
def test_ppo_update_matches_oracle(sharing, P, n_agents, clip, epochs, lr_):
    from codebase_b200.dqn.model import sharing_to_nets
    from codebase_b200.lbf import TrajStore

    rng = np.random.default_rng(P + epochs)
    hp = lr.A2CHP(grad_clip=clip, lr=lr_, target_update_interval_or_tau=2)
    m = _model(sharing, hp, P, n_agents, epochs, 0.2)
    nets = sharing_to_nets(sharing, n_agents)
    st = lr.A2CState(m.theta[: m.n_actor].cpu().clone(), m.theta[m.n_actor:].cpu().clone(), m.theta_tgt.cpu().clone(), nets, nets, D, A)
    for u, step in enumerate((0, 3, 4)):
        s = _batch_arrays(rng, P, n_agents)
        want = lr.ppo_update(st, _oracle_batch(s), hp, step, epochs, 0.2)
        ts = TrajStore(P, n_agents, T, D, m.device)
        for k in ("obs", "act", "rew", "done", "filled"):
            getattr(ts, k).copy_(torch.as_tensor(s[k]))
        met = m.metrics_dict(m.update_from_store(ts, P, step))
        _close([met["loss"], met["actor_loss"], met["value_loss"], met["entropy"]], [want["loss"], want["actor_loss"], want["value_loss"], want["entropy"]], rtol=2e-5, atol=2e-5)
        d = np.abs(m.theta.cpu().numpy() - np.concatenate([st.actor.numpy(), st.critic.numpy()]))
        assert np.quantile(d, 0.999) < 1e-5 * max(1.0, lr_ / 3e-4) and d.max() < 2 * hp.lr * epochs * (u + 1) + 1e-6, (np.quantile(d, 0.999), d.max())
        assert np.quantile(np.abs(m.theta_tgt.cpu().numpy() - st.target.numpy()), 0.999) < 1e-5 * max(1.0, lr_ / 3e-4)
        # keep the two trajectories glued so that later updates compare like for like
        m.theta.copy_(torch.cat([st.actor, st.critic])); m.theta_tgt.copy_(st.target)
        m.adam_m.copy_(torch.cat([st.m["actor"], st.m["critic"]])); m.adam_v.copy_(torch.cat([st.v["actor"], st.v["critic"]]))


@pytest.mark.gpu
@pytest.mark.parametrize("cls", ["A2CNetwork", "PPONetwork"])
def test_standardise_returns_matches_oracle(cls):
    """cfg.standardise_returns=True on the device (marl_a2c_standardise_returns): metrics, running statistics and parameters against the oracle"""
    from codebase_b200.lbf import TrajStore

    P, n_agents, epochs = 200, 2, 3
    rng = np.random.default_rng(21)
    hp = lr.A2CHP(target_update_interval_or_tau=2)
    m = _model(False, hp, P, n_agents, epochs, 0.2, standardise=True, cls=cls)
    st = lr.A2CState(m.theta[: m.n_actor].cpu().clone(), m.theta[m.n_actor:].cpu().clone(), m.theta_tgt.cpu().clone(), [0, 1], [0, 1], D, A,
                     ret_ms=lr.RunningMeanStdRef((n_agents,)))
    for u, step in enumerate((0, 2, 5)):
        s = _batch_arrays(rng, P, n_agents)
        s["rew"] *= 3.0   # returns away from the unit scale the statistics start at
        want = lr.ppo_update(st, _oracle_batch(s), hp, step, epochs, 0.2) if cls == "PPONetwork" else lr.a2c_update(st, _oracle_batch(s), hp, step)
        ts = TrajStore(P, n_agents, T, D, m.device)
        for k in ("obs", "act", "rew", "done", "filled"):
            getattr(ts, k).copy_(torch.as_tensor(s[k]))
        met = m.metrics_dict(m.update_from_store(ts, P, step))
        _close([met["loss"], met["actor_loss"], met["value_loss"], met["entropy"]], [want["loss"], want["actor_loss"], want["value_loss"], want["entropy"]], rtol=2e-5, atol=2e-5)
        mean, var, count = m.ret_ms()
        _close(mean.numpy(), st.ret_ms.mean.numpy()); _close(var.numpy(), st.ret_ms.var.numpy()); assert abs(count - st.ret_ms.count) < 1e-6
        _, ret, _ = m.scratch(P, T)
        _close(ret.permute(2, 1, 0).cpu().numpy(), want["returns"].numpy(), rtol=2e-5, atol=2e-5)
        d = np.abs(m.theta.cpu().numpy() - np.concatenate([st.actor.numpy(), st.critic.numpy()]))
        assert np.quantile(d, 0.999) < 1e-5, (u, np.quantile(d, 0.999))
        m.theta.copy_(torch.cat([st.actor, st.critic])); m.theta_tgt.copy_(st.target)
        m.adam_m.copy_(torch.cat([st.m["actor"], st.m["critic"]])); m.adam_v.copy_(torch.cat([st.v["actor"], st.v["critic"]]))


@pytest.mark.gpu
@pytest.mark.parametrize("cls,sharing", [("A2CNetwork", False), ("PPONetwork", True)])
def test_centralised_critic_matches_oracle(cls, sharing):
    """MAA2C / MAPPO on the device: the critic passes read the joint observation rows (source mode 2; `values()`: mode 3)"""
    from codebase_b200.lbf import TrajStore

    P, n_agents, epochs = 300, 2, 2
    rng = np.random.default_rng(31)
    hp = lr.A2CHP(target_update_interval_or_tau=2)
    m = _model(sharing, hp, P, n_agents, epochs, 0.2, cls=cls, centralised=True)
    nets = [0, 0] if sharing else [0, 1]
    assert m.n_critic == len(set(nets)) * lr.net_size(n_agents * D, 1)
    st = lr.A2CState(m.theta[: m.n_actor].cpu().clone(), m.theta[m.n_actor:].cpu().clone(), m.theta_tgt.cpu().clone(), nets, nets, D, A, centralised=True)
    obs = rng.integers(-1, 8, size=(77, n_agents, D)).astype(np.float32)
    joint = torch.tensor(obs.reshape(77, n_agents * D))
    want_v = torch.cat(lr.agents_forward(st.critic, nets, [joint] * n_agents, n_agents * D, 1), -1).numpy()
    _close(m.values(torch.tensor(obs, device="cuda")).cpu().numpy(), want_v)
    for u, step in enumerate((0, 2, 5)):
        s = _batch_arrays(rng, P, n_agents)
        want = lr.ppo_update(st, _oracle_batch(s), hp, step, epochs, 0.2) if cls == "PPONetwork" else lr.a2c_update(st, _oracle_batch(s), hp, step)
        ts = TrajStore(P, n_agents, T, D, m.device)
        for k in ("obs", "act", "rew", "done", "filled"):
            getattr(ts, k).copy_(torch.as_tensor(s[k]))
        met = m.metrics_dict(m.update_from_store(ts, P, step))
        _close([met["loss"], met["actor_loss"], met["value_loss"], met["entropy"]], [want["loss"], want["actor_loss"], want["value_loss"], want["entropy"]], rtol=2e-5, atol=2e-5)
        d = np.abs(m.theta.cpu().numpy() - np.concatenate([st.actor.numpy(), st.critic.numpy()]))
        assert np.quantile(d, 0.999) < 1e-5, (u, np.quantile(d, 0.999))
        m.theta.copy_(torch.cat([st.actor, st.critic])); m.theta_tgt.copy_(st.target)
        m.adam_m.copy_(torch.cat([st.m["actor"], st.m["critic"]])); m.adam_v.copy_(torch.cat([st.v["actor"], st.v["critic"]]))
    sd = m.state_dict()
    assert sd["critic." + ("networks" if sharing else "independent") + ".0.network.0.weight"].shape == (128, n_agents * D)


@pytest.mark.gpu
def test_ippo_driver_runs_and_logs(tmp_path, monkeypatch):
    """ac.train.main with +algorithm=ippo end to end: results.csv has the reference's AC columns"""
    import pandas as pd

    from codebase_b200 import run

    monkeypatch.chdir(tmp_path)
    run.main(["+algorithm=ippo", "env.name=lbforaging:Foraging-8x8-2p-3f-v3", "env.time_limit=25", "env.parallel_envs=256", "seed=1",
              "algorithm.total_steps=40000", "algorithm.eval_interval=10000", f"run_dir={tmp_path}/out"])
    df = pd.read_csv(tmp_path / "out" / "results.csv")
    for col in ("environment_steps", "actor_loss", "entropy", "value_loss", "loss", "mean_episode_returns", "updates"):
        assert col in df.columns, col
    assert len(df) >= 3 and df["environment_steps"].is_monotonic_increasing


@pytest.mark.gpu
@pytest.mark.parametrize("alg", ["maa2c", "mappo"])
def test_centralised_critic_drivers_run_and_log(tmp_path, monkeypatch, alg):
    """+algorithm=maa2c / mappo (critic.centralised: True) end to end on the 2-agent task whose joint observation (30) fits the kernels' 32 input features"""
    import pandas as pd

    from codebase_b200 import run

    monkeypatch.chdir(tmp_path)
    run.main([f"+algorithm={alg}", "env.name=lbforaging:Foraging-8x8-2p-3f-v3", "env.time_limit=25", "env.parallel_envs=256", "seed=2",
              "algorithm.total_steps=30000", "algorithm.eval_interval=10000", f"run_dir={tmp_path}/out"])
    df = pd.read_csv(tmp_path / "out" / "results.csv")
    assert len(df) >= 2 and np.isfinite(df["value_loss"].iloc[-1]) and df["environment_steps"].is_monotonic_increasing
