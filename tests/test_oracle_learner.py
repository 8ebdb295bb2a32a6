"""CPU: oracle/learner_ref.py (the torch-CPU restatement the GPU tests compare against) pinned against golden vectors
produced by the LIVE reference classes (tests/golden/make_golden.py, make_reference_cases below)."""
import os

import numpy as np
import pytest
import torch

from oracle import learner_ref as lr
from tests.helpers import load_case, net_layers, sample_index

GOLD = os.path.join(os.path.dirname(__file__), "golden")
N, D, A, T = 2, 15, 6, 25
RT, AT = 1e-5, 1e-5


def _close(a, b, rtol=RT, atol=AT):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert np.allclose(a, b, rtol=rtol, atol=atol), float(np.abs(a - b).max())


def _close_scaled(a, b, tol=1e-5):
    """element-wise, relative to the tensor's own scale (Adam's second moment lives at 1e-6 .. 1e-10: a plain atol would hide it).  For
    v = (1 - beta2) g^2 pass tol=2e-5: a relative gradient error e shows up as 2e in v, so 2e-5 on v is the 1e-5 bar on g."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    scale = max(float(np.abs(b).max()), 1e-30)
    assert np.abs(a - b).max() <= tol * scale, (float(np.abs(a - b).max()), scale)


def load_dqn_case(name):
    g = np.load(os.path.join(GOLD, f"{name}.npz"))
    hp = lr.DqnHP(lr=float(g["hp"][0]), gamma=float(g["hp"][1]), grad_clip=float(g["hp"][2]), double_q=bool(g["hp"][3]),
                  target_update_interval_or_tau=float(g["hp"][4]), mixer=int(g["mixer"]))
    return g, hp


@pytest.mark.parametrize("name", ["idqn_indep", "idqn_single_q_polyak_noclip", "idqn_shared", "vdn_indep"])
def test_dqn_update_matches_reference_golden(name):
    g, hp = load_dqn_case(name)
    theta = torch.tensor(g["theta0"])
    st = lr.DqnState(theta.clone(), theta.clone(), [int(x) for x in g["agent_net"]], D, A)
    for u in range(len(g["losses"])):
        store = {k: g[f"u{u}_{k}"] for k in ("obs", "act", "rew", "done", "filled")}
        out = lr.dqn_update(st, lr.batch_from_store(store, g[f"u{u}_idx"]), hp)
        _close(out["loss"], g["losses"][u])
        if u == 0:
            _close(out["grad"].numpy(), g["grad0"])
            _close_scaled(out["grad_clipped"].numpy(), g["grad0_clipped"])   # what Adam consumed (after clip_grad_norm_)
    _close_scaled(st.m.numpy(), g["adam_m_final"])   # element-wise: the loose bound on theta below cannot hide a defect here
    _close_scaled(st.v.numpy(), g["adam_v_final"], tol=2e-5)
    # Adam's first steps move every weight by ~lr regardless of |g|: elements whose gradient is rounding noise may
    # flip sign between two float32 summation orders, so compare the bulk tightly and bound the rest by 2*lr per step.
    d = np.abs(st.theta.numpy() - g["theta_final"])
    assert np.quantile(d, 0.999) < 1e-5 and d.max() < 2 * hp.lr * len(g["losses"]) + 1e-6
    _close(np.quantile(np.abs(st.theta_tgt.numpy() - g["target_final"]), 0.999), 0, atol=1e-5)


@pytest.mark.parametrize("name", ["ia2c_indep", "ia2c_shared"])
def test_a2c_update_matches_reference_golden(name):
    g = np.load(os.path.join(GOLD, f"{name}.npz"))
    hp = lr.A2CHP(lr=float(g["hp"][0]), gamma=float(g["hp"][1]), grad_clip=float(g["hp"][2]), n_steps=int(g["hp"][3]), entropy_coef=float(g["hp"][4]),
                  value_loss_coef=float(g["hp"][5]), target_update_interval_or_tau=float(g["hp"][6]))
    nets = [int(x) for x in g["agent_net"]]
    st = lr.A2CState(torch.tensor(g["actor0"]), torch.tensor(g["critic0"]), torch.tensor(g["target0"]), nets, nets, D, A)
    for u, step in enumerate(g["steps"]):
        s = {k: torch.as_tensor(g[f"u{u}_{k}"]) for k in ("obs", "act", "rew", "done", "filled")}
        P = s["obs"].shape[0]
        batch = dict(obss=s["obs"].permute(2, 0, 1, 3).reshape(T + 1, P, N * D).float(), actions=s["act"].permute(2, 0, 1).long(),
                     rewards=s["rew"].permute(2, 0, 1).float(), dones=s["done"].permute(1, 0).float(), filled=s["filled"].permute(1, 0).float())
        out = lr.a2c_update(st, batch, hp, int(step))
        _close([out["loss"], out["actor_loss"], out["value_loss"], out["entropy"]], g["metrics"][u])
        if u == 0:
            _close(out["returns"].numpy(), g["returns0"])
            for k in ("actor", "critic"):
                _close_scaled(out["grad_clipped"][k].numpy(), g[f"{k}_grad0_clipped"])
    for k in ("actor", "critic"):
        _close_scaled(st.m[k].numpy(), g[f"{k}_adam_m_final"])
        _close_scaled(st.v[k].numpy(), g[f"{k}_adam_v_final"], tol=2e-5)
    for mine, want in ((st.actor, "actor_final"), (st.critic, "critic_final"), (st.target, "target_final")):
        d = np.abs(mine.numpy() - g[want])
        assert np.quantile(d, 0.999) < 1e-5 and d.max() < 2 * hp.lr * len(g["steps"]) + 1e-6


def test_epsilon_schedule_and_nstep_returns_golden():
    g = np.load(os.path.join(GOLD, "misc.npz"))
    lin = lr.epsilon_schedule("linear", 0.5, 1.0, 0.05, 6.5, 100000)
    exp = lr.epsilon_schedule("exponential", 0.5, 1.0, 0.05, 6.5, 100000)
    assert np.array_equal(np.array([lin(int(s)) for s in g["steps"]]), g["eps_linear"])
    assert np.array_equal(np.array([exp(int(s)) for s in g["steps"]]), g["eps_exp"])
    for n in (1, 5, 30):
        got = lr.nstep_returns(torch.tensor(g["ns_rew"]), torch.tensor(g["ns_done"]), torch.tensor(g["ns_nv"]), n, 0.99)
        _close(got.numpy(), g[f"ns_ret_{n}"], rtol=1e-6, atol=1e-6)


LIVE = os.path.join(GOLD, "ref_oracle_learner.npz")


def _replay_episodes(rng):
    """12 episodes of random lengths into a 5-slot ring: (first observations, [(observations, actions, rewards, done) per step]) per episode"""
    for _ in range(12):
        L = int(rng.integers(2, T + 1))
        o0 = [rng.standard_normal(D).astype(np.float32) for _ in range(N)]
        steps = []
        for t in range(L):
            o = [rng.standard_normal(D).astype(np.float32) for _ in range(N)]
            steps.append((o, rng.integers(0, A, N), rng.random(N).astype(np.float32), t == L - 1))
        yield o0, steps


def _fresh_batch(rng, B=16):
    return dict(obss=torch.tensor(rng.standard_normal((N, T + 1, B, D)), dtype=torch.float32), actions=torch.tensor(rng.integers(0, A, (N, T, B))),
                rewards=torch.tensor(rng.random((N, T, B)), dtype=torch.float32), dones=torch.tensor(rng.random((T + 1, B)) < 0.05, dtype=torch.float32),
                filled=torch.tensor(rng.random((T, B)) < 0.9, dtype=torch.float32))


def make_reference_cases():
    """Records tests/golden/ref_oracle_learner.npz from the reference's ReplayBuffer and QNetwork: MARLBASE_SRC=<marlbase checkout> python -c 'import
    tests.test_oracle_learner as t; t.make_reference_cases()'."""
    from oracle import ref_shim

    ref = ref_shim.load()
    rb = ref.dqn_train.ReplayBuffer(5, N, [ref_shim.Space(shape=(D,)) for _ in range(N)], [ref_shim.Space(n=A)] * N, T, "cpu")
    for o0, steps in _replay_episodes(np.random.default_rng(1)):
        rb.init_episode(o0)
        for o, a, r, d in steps:
            rb.add(o, a, r, d)
    out = {"ring.len": np.int64(len(rb)), "ring.cur_pos": np.int64(rb.cur_pos), "ring.actions": rb.actions, "ring.rewards": rb.rewards,
           "ring.dones": rb.dones, "ring.filled": rb.filled, "ring.observations": np.stack(rb.observations)}
    torch.manual_seed(123)
    model = ref.dqn_model.QNetwork([ref_shim.Space(shape=(D,))] * N, [ref_shim.Space(n=A)] * N, ref_shim.dqn_cfg(), [128, 128], False, False, True, "cpu")
    idx = sample_index(net_layers(N, D, A))
    out["fresh.theta0"] = lr.flat_from_state_dict(model.state_dict(), "critic.independent", N).numpy()[idx]
    rng = np.random.default_rng(4)
    losses = []
    for _ in range(2):
        b = _fresh_batch(rng)
        losses.append(model.update(ref.dqn_train.Batch(b["obss"], b["actions"], b["rewards"], b["dones"], b["filled"], None))["loss"])
    out["fresh.loss"] = np.array(losses, np.float64)
    out["fresh.theta"] = lr.flat_from_state_dict(model.state_dict(), "critic.independent", N).numpy()[idx]
    np.savez_compressed(LIVE, **out)


def test_replay_ring_matches_live_reference_buffer():
    """ReplayRef (episode-major) == reference ReplayBuffer (time-major, recorded in tests/golden/ref_oracle_learner.npz) incl. the stale tail of
    re-used slots."""
    rb = load_case(LIVE, "ring")
    mine = lr.ReplayRef(5, N, T, D)
    for o0, steps in _replay_episodes(np.random.default_rng(1)):
        mine.init_episode(o0)
        for o, a, r, d in steps:
            mine.add(o, a, r, d)
    assert int(rb["len"]) == len(mine) and int(rb["cur_pos"]) == mine.cur
    for i in range(N):
        assert np.array_equal(rb["observations"][i].transpose(1, 0, 2), mine.store["obs"][:, i])
    assert np.array_equal(rb["actions"].transpose(2, 0, 1), mine.store["act"])
    assert np.array_equal(rb["rewards"].transpose(2, 0, 1), mine.store["rew"])
    assert np.array_equal(rb["dones"].T, mine.store["done"].astype(bool)) and np.array_equal(rb["filled"].T, mine.store["filled"].astype(bool))


def test_live_reference_update_on_fresh_seed():
    """Not only the fixtures of make_golden.py: a further random case (the reference's default DQN settings, torch seed 123) against what the
    reference's QNetwork computed (tests/golden/ref_oracle_learner.npz)."""
    g = load_case(LIVE, "fresh")
    idx = sample_index(net_layers(N, D, A))
    torch.manual_seed(123)
    theta = lr.init_flat(N, D, A)
    assert np.abs(theta.numpy()[idx] - g["theta0"]).max() < 1e-6, "initialisation differs from the reference's"
    st = lr.DqnState(theta.clone(), theta.clone(), [0, 1], D, A)
    rng = np.random.default_rng(4)
    for want in g["loss"]:
        got = lr.dqn_update(st, _fresh_batch(rng), lr.DqnHP())
        _close(got["loss"], want)
    d = np.abs(st.theta.numpy()[idx] - g["theta"])
    assert np.quantile(d, 0.999) < 1e-5


@pytest.mark.parametrize("alg", ["ia2c", "mappo"])
def test_cpu_actor_critic_loop_collects_the_reference_batch_layout(alg):
    """oracle/cpu_loop_ac.py (the CPU arm of tools/learning_curve_ac.py): one iteration fills a Batch as ac/train.py:24-119 does -- obs row 0 from
    reset, `filled` a prefix of ones per env, the done flag of the last filled step set, nothing written after an env finished -- and the update moves
    the parameters."""
    from oracle.cpu_loop_ac import CpuAC
    from oracle.lbf_ref import LBFConfig

    loop = CpuAC(alg, LBFConfig(time_limit=6), parallel_envs=5, seed=3)
    t, b, infos = loop.collect()
    assert 1 <= t <= 6 and len(infos) == 5 and all("episode_returns" in i for i in infos)
    filled = b["filled"].numpy()
    for i in range(5):
        L = int(filled[:, i].sum())
        assert L >= 1 and (filled[:L, i] == 1).all() and (filled[L:, i] == 0).all()
        assert b["dones"][L, i] == 1 and (b["dones"][:L, i] == 0).all()
        assert (b["obss"][L + 1:, i] == 0).all() and (b["rewards"][L:, i] == 0).all() and (b["actions"][L:, i] == 0).all()
        assert (b["obss"][: L + 1, i] != 0).any()
    before = loop.st.actor.clone()
    at, ret = loop.iteration()
    assert at == 0 and loop.step == loop.P * max(1, int(loop.step / loop.P)) and np.isfinite(ret) and not torch.equal(before, loop.st.actor)
