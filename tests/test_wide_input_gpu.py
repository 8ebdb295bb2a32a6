"""GPU: input widths 33..128 (K-chunked first layer of the FP32 learner kernels) -- IDQN / VDN / QMIX updates and q_values, IA2C / IPPO, and the
centralised critics of MAA2C / MAPPO (4 agents x 27 or 31 features: 108 / 124 wide) against the CPU oracle; narrow learners unaffected by wide ones;
the drivers end to end on Foraging-20x20-9p-6f (45 features, 9 agents) and Foraging-15x15-4p-5f (centralised critic of 108)."""
import types

import numpy as np
import pytest
import torch

from oracle import learner_ref as lr
from oracle import qmix_ref as qr
from tests.helpers import NearTie, assert_grad_close, check_margin, redraw_on_near_tie

pytestmark = pytest.mark.gpu
A = 6


def _close(a, b, rtol=1e-5, atol=1e-5):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert np.allclose(a, b, rtol=rtol, atol=atol), float(np.abs(a - b).max())


def _space(shape=None, n=None):
    return types.SimpleNamespace(shape=shape, n=n)


def _random_store(rng, cap, n_agents, D, T, coop):
    obs = rng.integers(-1, 15, size=(cap, n_agents, T + 1, D)).astype(np.float32)
    act = rng.integers(0, A, size=(cap, n_agents, T)).astype(np.int32)
    rew = (rng.random((cap, n_agents, T)) < 0.2).astype(np.float32) * rng.random((cap, n_agents, T)).astype(np.float32)
    if coop:
        rew[:] = rew[:, :1]
    length = rng.integers(1, T + 1, size=cap)
    done = np.zeros((cap, T + 1), np.uint8); filled = np.zeros((cap, T), np.uint8)
    for e in range(cap):
        filled[e, : length[e]] = 1
        done[e, length[e]] = 1
    return dict(obs=obs, act=act, rew=rew, done=done, filled=filled)


def _to_store(s, device):
    from codebase_b200.lbf import TrajStore

    cap, n_agents, T1, D = s["obs"].shape
    ts = TrajStore(cap, n_agents, T1 - 1, D, device)
    for k in ("obs", "act", "rew", "done", "filled"):
        getattr(ts, k).copy_(torch.as_tensor(s[k]))
    return ts


def _dqn_model(mixer, sharing, n_agents, D, B, T, hp):
    from codebase_b200.dqn import model as M

    cfg = types.SimpleNamespace(optimizer="Adam", lr=hp.lr, gamma=hp.gamma, grad_clip=hp.grad_clip, double_q=hp.double_q,
                                target_update_interval_or_tau=hp.target_update_interval_or_tau, standardise_returns=False)
    spaces = ([_space(shape=(D,))] * n_agents, [_space(n=A)] * n_agents)
    if mixer == 2:
        return M.QMixNetwork(*spaces, cfg, [128, 128], sharing, False, True, dict(embed_dim=64, hypernet_layers=2, hypernet_embed=32), "cuda",
                             max_batch=B, max_episode_length=T)
    return (M.VDNetwork if mixer else M.QNetwork)(*spaces, cfg, [128, 128], sharing, False, True, "cuda", max_batch=B, max_episode_length=T)


def _q_values_match(m, rng, n_agents, D):
    """q_values on dense rows (tensor_core_forward left on: a wide network must take the FFMA kernels) against the oracle"""
    obs = rng.integers(-1, 15, size=(50, n_agents, D)).astype(np.float32)
    want = torch.stack(lr.agents_forward(m.theta.cpu(), m.agent_net, [torch.tensor(obs[:, i]) for i in range(n_agents)], D, A), 1).numpy()
    _close(m.q_values(torch.tensor(obs, device="cuda")).cpu().numpy(), want)


# (mixer, parameter sharing, agents, width, batch, T): 0 = IDQN, 1 = VDN, 2 = QMIX (its mixer and a 32-sample tile must fit shared memory: state
# N x D = 128 does); batches whose rows end in ragged tiles
DQN_CASES = [(0, False, 2, 33, 40, 7), (0, True, 3, 45, 130, 25), (1, [0, 1, 0], 3, 64, 33, 7), (0, False, 2, 65, 50, 25), (1, False, 2, 100, 21, 25),
             (0, [0, 1, 0], 3, 128, 77, 7), (2, False, 2, 45, 16, 7), (2, True, 2, 64, 33, 25)]


@pytest.mark.parametrize("mixer,sharing,n_agents,D,B,T", DQN_CASES)
@redraw_on_near_tie
def test_dqn_family_update_at_wide_obs(mixer, sharing, n_agents, D, B, T):
    from codebase_b200.dqn.model import sharing_to_nets

    rng = np.random.default_rng(D * 1000 + B)
    hp = lr.DqnHP(mixer=1 if mixer == 1 else 0, target_update_interval_or_tau=2.0)   # (QMIX: the oracle's mixer is qmix_ref's)
    m = _dqn_model(mixer, sharing, n_agents, D, B, T, hp)
    agent_net = sharing_to_nets(sharing, n_agents)
    _q_values_match(m, rng, n_agents, D)
    store = _random_store(rng, 200, n_agents, D, T, mixer > 0)
    idx = rng.integers(0, 200, size=B).astype(np.int32)
    batch = lr.batch_from_store(store, idx)
    st = lr.DqnState(m.theta.cpu().clone(), m.theta_tgt.cpu().clone(), agent_net, D, A)
    check_margin(lr, st, batch, hp)   # near-tie in the double-Q argmax: re-drawn by the decorator
    if mixer == 2:
        qs = qr.QmixState(m.theta.cpu().clone(), m.theta_tgt.cpu().clone(), m.mix.cpu().clone(), m.mix_tgt.cpu().clone(), agent_net, D, A)
        qs0 = qr.QmixState(qs.theta.clone(), qs.theta_tgt.clone(), qs.mix.clone(), qs.mix_tgt.clone(), agent_net, D, A)
        want = qr.qmix_update(qs, batch, hp)
        met = m.update_from_store(_to_store(store, m.device), torch.tensor(idx, device="cuda")).cpu()
        filled = float(batch["filled"].sum())
        got = m.grad[: m.n_params].cpu().numpy() / filled
        err = float(np.abs(got - want["grad"].numpy()).max())
        if err > 2e-5 * max(1.0, float(want["grad"].abs().max())):
            if qr.qmix_kink_risk(qs0, batch, hp) >= 0.5 * err:
                raise NearTie()
            raise AssertionError(f"agents' gradient: max abs error {err:.3e}")
        assert abs(float(met[0]) - want["loss"]) <= 1e-5 * max(1.0, abs(want["loss"]))
        for mine, theirs, what in ((m.theta, qs.theta, "theta"), (m.mix, qs.mix, "mixer"), (m.theta_tgt, qs.theta_tgt, "target")):
            assert np.quantile(np.abs(mine.cpu().numpy() - theirs.numpy()), 0.999) < 2e-5, what
    else:
        st0 = lr.DqnState(st.theta.clone(), st.theta_tgt.clone(), agent_net, D, A)   # dqn_update steps st in place
        want = lr.dqn_update(st, batch, hp)
        m.update_grads(_to_store(store, m.device), torch.tensor(idx, device="cuda"))
        gr = m.grad.cpu().numpy()
        assert_grad_close(lr, st0, batch, hp, gr[: m.n_params] / gr[m.n_params + 1], want["grad"].numpy())
        _close(m.update_apply().cpu().numpy()[0], want["loss"])
        assert np.quantile(np.abs(m.theta.cpu().numpy() - st.theta.numpy()), 0.999) < 1e-5
    _q_values_match(m, rng, n_agents, D)   # the forward after Adam: no stale tensor-core image may be used for the wide network
    m.close()


@redraw_on_near_tie
def test_three_consecutive_updates_at_45_features():
    """Three fused updates in a row (marl_dqn_update: forward, train pass, reduce + Adam, hard target copy after the second) against the oracle's"""
    n_agents, D, B, T = 3, 45, 64, 25
    rng = np.random.default_rng(45)
    hp = lr.DqnHP(target_update_interval_or_tau=2.0)
    m = _dqn_model(0, False, n_agents, D, B, T, hp)
    st = lr.DqnState(m.theta.cpu().clone(), m.theta_tgt.cpu().clone(), m.agent_net, D, A)
    store = _random_store(rng, 200, n_agents, D, T, False)
    ts = _to_store(store, m.device)
    for u in range(3):
        idx = rng.integers(0, 200, size=B).astype(np.int32)
        batch = lr.batch_from_store(store, idx)
        check_margin(lr, st, batch, hp)
        want = lr.dqn_update(st, batch, hp)
        loss = float(m.update_from_store(ts, torch.tensor(idx, device="cuda"))[0].item())
        assert abs(loss - want["loss"]) <= 1e-5 * max(1.0, abs(want["loss"])), u
        assert np.quantile(np.abs(m.theta.cpu().numpy() - st.theta.numpy()), 0.999) < 1e-5, u
        assert np.quantile(np.abs(m.theta_tgt.cpu().numpy() - st.theta_tgt.numpy()), 0.999) < 1e-5, u
    _q_values_match(m, rng, n_agents, D)
    m.close()


def test_observation_wider_than_128_is_refused():
    from codebase_b200.dqn import model as M

    cfg = types.SimpleNamespace(optimizer="Adam", lr=3e-4, gamma=0.99, grad_clip=1.0, double_q=True, target_update_interval_or_tau=200, standardise_returns=False)
    with pytest.raises(NotImplementedError, match="129 wide"):
        M.QNetwork([_space(shape=(129,))] * 2, [_space(n=A)] * 2, cfg, [128, 128], False, False, True, "cuda", max_batch=8, max_episode_length=5)


# ---- actor-critic ---------------------------------------------------------------------------------------------------------------------------------
def _ac_model(cls, sharing, centralised, n_agents, D, P, T, hp, epochs=2):
    from codebase_b200.ac import model as M

    cfg = types.SimpleNamespace(optimizer="Adam", lr=hp.lr, gamma=hp.gamma, grad_clip=hp.grad_clip, n_steps=hp.n_steps, entropy_coef=hp.entropy_coef,
                                value_loss_coef=hp.value_loss_coef, target_update_interval_or_tau=hp.target_update_interval_or_tau, standardise_returns=False,
                                num_epochs=epochs, ppo_clip=0.2)
    net = types.SimpleNamespace(layers=[128, 128], parameter_sharing=sharing, use_rnn=False, use_orthogonal_init=True, centralised=False)
    cnet = types.SimpleNamespace(layers=[128, 128], parameter_sharing=sharing, use_rnn=False, use_orthogonal_init=True, centralised=centralised)
    return getattr(M, cls)([_space(shape=(D,))] * n_agents, [_space(n=A)] * n_agents, cfg, net, cnet, "cuda", max_envs=P, max_episode_length=T)


def _oracle_ac_batch(s):
    t = {k: torch.as_tensor(v) for k, v in s.items()}
    P, n_agents, T1, D = t["obs"].shape
    return dict(obss=t["obs"].permute(2, 0, 1, 3).reshape(T1, P, n_agents * D).float(), actions=t["act"].permute(2, 0, 1).long(),
                rewards=t["rew"].permute(2, 0, 1).float(), dones=t["done"].permute(1, 0).float(), filled=t["filled"].permute(1, 0).float())


# (class, parameter sharing, centralised critic, agents, width, envs): IA2C / IPPO at 45 features; MAA2C / MAPPO with critics of 108 and 124
AC_CASES = [("A2CNetwork", False, False, 3, 45, 96), ("PPONetwork", True, False, 3, 45, 150), ("A2CNetwork", False, True, 4, 27, 100),
            ("PPONetwork", True, True, 4, 27, 64), ("A2CNetwork", True, True, 4, 31, 80), ("PPONetwork", False, True, 4, 31, 120)]


@pytest.mark.parametrize("cls,sharing,centralised,n_agents,D,P", AC_CASES)
def test_actor_critic_update_at_wide_obs(cls, sharing, centralised, n_agents, D, P):
    from codebase_b200.dqn.model import sharing_to_nets

    T, epochs = 25, 2
    rng = np.random.default_rng(D * 100 + P)
    hp = lr.A2CHP(target_update_interval_or_tau=2)
    m = _ac_model(cls, sharing, centralised, n_agents, D, P, T, hp, epochs)
    nets = sharing_to_nets(sharing, n_agents)
    c_in = n_agents * D if centralised else D
    assert m.n_critic == len(set(nets)) * lr.net_size(c_in, 1)
    st = lr.A2CState(m.theta[: m.n_actor].cpu().clone(), m.theta[m.n_actor:].cpu().clone(), m.theta_tgt.cpu().clone(), nets, nets, D, A, centralised=centralised)
    obs = rng.integers(-1, 8, size=(77, n_agents, D)).astype(np.float32)
    xs = [torch.tensor(obs.reshape(77, n_agents * D))] * n_agents if centralised else [torch.tensor(obs[:, i]) for i in range(n_agents)]
    _close(m.values(torch.tensor(obs, device="cuda")).cpu().numpy(), torch.cat(lr.agents_forward(st.critic, nets, xs, c_in, 1), -1).numpy())
    for u, step in enumerate((0, 2, 5)):
        s = _random_store(rng, P, n_agents, D, T, False)
        b = _oracle_ac_batch(s)
        want = lr.ppo_update(st, b, hp, step, epochs, 0.2) if cls == "PPONetwork" else lr.a2c_update(st, b, hp, step)
        met = m.metrics_dict(m.update_from_store(_to_store(s, m.device), P, step))
        _close([met[k] for k in ("loss", "actor_loss", "value_loss", "entropy")], [want[k] for k in ("loss", "actor_loss", "value_loss", "entropy")], rtol=2e-5, atol=2e-5)
        d = np.abs(m.theta.cpu().numpy() - np.concatenate([st.actor.numpy(), st.critic.numpy()]))
        assert np.quantile(d, 0.999) < 1e-5, (u, np.quantile(d, 0.999))
        # keep the two trajectories glued so that later updates compare like for like
        m.theta.copy_(torch.cat([st.actor, st.critic])); m.theta_tgt.copy_(st.target)
        m.adam_m.copy_(torch.cat([st.m["actor"], st.m["critic"]])); m.adam_v.copy_(torch.cat([st.v["actor"], st.v["critic"]]))
    m.close()


def test_centralised_critic_wider_than_128_is_refused():
    hp = lr.A2CHP()
    with pytest.raises(NotImplementedError, match="129 wide"):
        _ac_model("A2CNetwork", False, True, 3, 43, 16, 5, hp)


# ---- the narrow path is untouched; the wide path is deterministic ---------------------------------------------------------------------------------
def _one_update(D, seed, B=96, T=25, n_agents=3):
    torch.manual_seed(seed)
    hp = lr.DqnHP()
    m = _dqn_model(1, False, n_agents, D, B, T, hp)
    rng = np.random.default_rng(seed)
    store = _random_store(rng, 200, n_agents, D, T, True)
    idx = torch.tensor(rng.integers(0, 200, size=B).astype(np.int32), device="cuda")
    ts = _to_store(store, m.device)
    m.update_from_store(ts, idx)
    m.update_from_store(ts, idx)
    out = (m.theta.cpu().clone(), m.q_values(ts.obs[:8, :, 0].contiguous()).cpu().clone())
    m.close()
    return out


def test_narrow_learner_bit_identical_around_a_wide_one():
    """A 27-feature VDN learner (tensor-core forward and training pass) computes the same bits before and after a 45-feature learner was created and
    updated in the same process (shared-memory opt-in and tensor-core dispatch are per network); two runs of the wide learner are bit-identical."""
    before = _one_update(27, 3)
    wide1 = _one_update(45, 4)
    after = _one_update(27, 3)
    wide2 = _one_update(45, 4)
    for x, y in zip(before, after):
        assert torch.equal(x, y)
    for x, y in zip(wide1, wide2):
        assert torch.equal(x, y)


# ---- the drivers end to end -----------------------------------------------------------------------------------------------------------------------
def test_idqn_driver_on_20x20_9p_6f_with_eval_round_trip(tmp_path, monkeypatch):
    """+algorithm=idqn on Foraging-20x20-9p-6f-v3 (9 agents x 45 features): results.csv with finite losses, then a checkpoint evaluated"""
    import os

    import pandas as pd

    from codebase_b200 import eval as ev
    from codebase_b200 import run

    monkeypatch.chdir(tmp_path)
    out = f"{tmp_path}/out"
    run.main(["+algorithm=idqn", "env.name=lbforaging:Foraging-20x20-9p-6f-v3", "env.time_limit=25", "env.parallel_envs=256", "seed=0",
              "algorithm.total_steps=40000", "algorithm.eval_interval=10000", "algorithm.save_interval=15000", "algorithm.batch_size=128",
              "algorithm.buffer_size=2048", "algorithm.updates_per_iteration=8", f"run_dir={out}"])
    df = pd.read_csv(f"{out}/results.csv")
    assert "agent8/mean_episode_returns" in df.columns and len(df) >= 2 and np.isfinite(df["loss"].iloc[-1])
    monkeypatch.chdir(tmp_path)
    steps = sorted(int(f[7:-3]) for f in os.listdir(f"{out}/checkpoints"))
    res = ev.main([f"path={out}", "episodes=32", "seed=3"])
    assert res["load_step"] == steps[-1] and res["episodes"] == 32 and np.isfinite(res["mean_episode_returns"])


def test_mappo_driver_on_15x15_4p_5f(tmp_path, monkeypatch):
    """+algorithm=mappo on Foraging-15x15-4p-5f-v3: the centralised critic reads 4 x 27 = 108 features"""
    import pandas as pd

    from codebase_b200 import run

    monkeypatch.chdir(tmp_path)
    run.main(["+algorithm=mappo", "env.name=lbforaging:Foraging-15x15-4p-5f-v3", "env.time_limit=25", "env.parallel_envs=256", "seed=2",
              "algorithm.total_steps=30000", "algorithm.eval_interval=10000", f"run_dir={tmp_path}/out"])
    df = pd.read_csv(tmp_path / "out" / "results.csv")
    assert len(df) >= 2 and np.isfinite(df["value_loss"].iloc[-1]) and np.isfinite(df["loss"].iloc[-1]) and df["environment_steps"].is_monotonic_increasing
