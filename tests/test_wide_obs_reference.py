"""CPU: the oracle (oracle/learner_ref.py, oracle/qmix_ref.py) at input widths 33..128 against recorded runs of the reference's classes
(tests/golden/ref_wide_obs.npz): a shared QNetwork on 9 agents x 45 features (Foraging-20x20-9p-6f), a QMixNetwork on 2 x 64 features (state 128),
and centralised critics of 4 x 27 = 108 (Foraging-15x15-4p-5f) and 4 x 31 = 124 (the same with observe_id) features."""
import os

import numpy as np
import pytest
import torch

from oracle import learner_ref as lr
from oracle import qmix_ref as qr
from tests.helpers import load_case, net_layers, sample_index

LIVE = os.path.join(os.path.dirname(__file__), "golden", "ref_wide_obs.npz")
A, T = 6, 10
METRICS = ("loss", "actor_loss", "value_loss", "entropy")
# name -> (class, n_agents, obs width, parameter sharing, torch seed, batch seed, batch size, config)
DQN_CASES = {
    "qnet_shared_9x45": ("QNetwork", 9, 45, True, 21, 4, 8, dict(target_update_interval_or_tau=2)),
    "qmix_2x64": ("QMixNetwork", 2, 64, False, 11, 5, 16, dict(target_update_interval_or_tau=2)),
}
# name -> (class, n_agents, obs width, parameter sharing, torch seed, batch seed, envs per batch, update steps, config)
AC_CASES = {
    "ppo_cent_4x27": ("PPONetwork", 4, 27, False, 4, 5, 10, (0, 2, 3), dict(num_epochs=3, ppo_clip=0.2, target_update_interval_or_tau=2)),
    "a2c_cent_shared_4x31": ("A2CNetwork", 4, 31, True, 6, 7, 10, (0, 2, 3), dict(target_update_interval_or_tau=2)),
}


def _dqn_batch(rng, n, d, B, coop):
    rew = rng.random((1 if coop else n, T, B))
    return dict(obss=torch.tensor(rng.standard_normal((n, T + 1, B, d)), dtype=torch.float32), actions=torch.tensor(rng.integers(0, A, (n, T, B))),
                rewards=torch.tensor(np.broadcast_to(rew, (n, T, B)).copy(), dtype=torch.float32),
                dones=torch.tensor(rng.random((T + 1, B)) < 0.05, dtype=torch.float32), filled=torch.tensor(rng.random((T, B)) < 0.9, dtype=torch.float32))


def _ac_batch(rng, P, n, d):
    obs = rng.integers(-1, 8, size=(P, n, T + 1, d)).astype(np.float32)
    act = rng.integers(0, A, size=(P, n, T))
    rew = (rng.random((P, n, T)) < 0.2).astype(np.float32) * rng.random((P, n, T)).astype(np.float32)
    length = rng.integers(1, T + 1, size=P)
    done = np.zeros((P, T + 1), np.float32); filled = np.zeros((P, T), np.float32)
    for e in range(P):
        filled[e, : length[e]] = 1
        done[e, length[e]] = 1
    return dict(obss=torch.tensor(obs).permute(2, 0, 1, 3).reshape(T + 1, P, n * d), actions=torch.tensor(act).permute(2, 0, 1),
                rewards=torch.tensor(rew).permute(2, 0, 1), dones=torch.tensor(done).T.contiguous(), filled=torch.tensor(filled).T.contiguous())


def _dqn_index(case):
    cls, n, d, sharing = DQN_CASES[case][:4]
    it = sample_index(net_layers(1 if sharing else n, d, A))
    return it, (sample_index(qr.mixer_shapes(n, n * d, 64, 32)) if cls == "QMixNetwork" else None)


def _ac_index(case):
    _, n, d, sharing = AC_CASES[case][:4]
    n_nets = 1 if sharing else n
    return sample_index(net_layers(n_nets, d, A)), sample_index(net_layers(n_nets, n * d, 1))


def make_reference_cases():
    """Records tests/golden/ref_wide_obs.npz from the reference's QNetwork, QMixNetwork, PPONetwork and A2CNetwork: MARLBASE_SRC=<marlbase checkout>
    python -c 'import tests.test_wide_obs_reference as t; t.make_reference_cases()'.  Per case: the losses (metrics) of each update and the parameters
    before and after at up to 64 evenly spaced positions per weight and bias."""
    from collections import namedtuple

    from oracle import ref_shim

    ref = ref_shim.load()
    AcBatch = namedtuple("Batch", ["obss", "actions", "rewards", "dones", "filled", "action_masks"])
    out = {}
    for case, (cls, n, d, sharing, seed, bseed, B, kw) in DQN_CASES.items():
        kind, n_nets = ("networks", 1) if sharing else ("independent", n)
        it, im = _dqn_index(case)
        torch.manual_seed(seed)
        cfg = ref_shim.dqn_cfg(**kw)
        spaces = ([ref_shim.Space(shape=(d,))] * n, [ref_shim.Space(n=A)] * n)
        if cls == "QMixNetwork":
            model = ref.dqn_model.QMixNetwork(*spaces, cfg, [128, 128], sharing, False, True, dict(embed_dim=64, hypernet_layers=2, hypernet_embed=32), "cpu")
        else:
            model = ref.dqn_model.QNetwork(*spaces, cfg, [128, 128], sharing, False, True, "cpu")
        sd = model.state_dict()
        out[f"{case}.theta0"] = lr.flat_from_state_dict(sd, f"critic.{kind}", n_nets).numpy()[it]
        if im is not None:
            out[f"{case}.mix0"] = qr.mixer_flat_from_state_dict(sd, "mixer").numpy()[im]
        rng = np.random.default_rng(bseed)
        losses = []
        for _ in range(3):
            b = _dqn_batch(rng, n, d, B, cls == "QMixNetwork")
            losses.append(model.update(ref.dqn_train.Batch(b["obss"], b["actions"], b["rewards"], b["dones"], b["filled"], None))["loss"])
        sd = model.state_dict()
        out.update({f"{case}.loss": np.array(losses, np.float64), f"{case}.theta": lr.flat_from_state_dict(sd, f"critic.{kind}", n_nets).numpy()[it],
                    f"{case}.theta_tgt": lr.flat_from_state_dict(sd, f"target.{kind}", n_nets).numpy()[it]})
        if im is not None:
            out.update({f"{case}.mix": qr.mixer_flat_from_state_dict(sd, "mixer").numpy()[im], f"{case}.mix_tgt": qr.mixer_flat_from_state_dict(sd, "target_mixer").numpy()[im]})
    for case, (cls, n, d, sharing, seed, bseed, P, steps, kw) in AC_CASES.items():
        kind, n_nets = ("networks", 1) if sharing else ("independent", n)
        ia, ic = _ac_index(case)
        torch.manual_seed(seed)
        model = getattr(ref.ac_model, cls)([ref_shim.Space(shape=(d,))] * n, [ref_shim.Space(n=A)] * n, ref_shim.a2c_cfg(**kw), ref_shim.net_cfg(parameter_sharing=sharing),
                                           ref_shim.net_cfg(parameter_sharing=sharing, centralised=True), "cpu")
        sd = model.state_dict()
        out[f"{case}.critic_in"] = np.int64(sd[f"critic.{kind}.0.network.0.weight"].shape[1])
        out[f"{case}.actor0"] = lr.flat_from_state_dict(sd, f"actor.{kind}", n_nets).numpy()[ia]
        out[f"{case}.critic0"] = lr.flat_from_state_dict(sd, f"critic.{kind}", n_nets).numpy()[ic]
        rng = np.random.default_rng(bseed)
        metrics = []
        for step in steps:
            b = _ac_batch(rng, P, n, d)
            got = model.update(AcBatch(b["obss"], b["actions"], b["rewards"], b["dones"].bool(), b["filled"], None), step)
            metrics.append([got[k] for k in METRICS])
        sd = model.state_dict()
        out.update({f"{case}.metrics": np.array(metrics, np.float64), f"{case}.actor": lr.flat_from_state_dict(sd, f"actor.{kind}", n_nets).numpy()[ia],
                    f"{case}.critic": lr.flat_from_state_dict(sd, f"critic.{kind}", n_nets).numpy()[ic],
                    f"{case}.target": lr.flat_from_state_dict(sd, f"target_critic.{kind}", n_nets).numpy()[ic]})
    np.savez_compressed(LIVE, **out)


@pytest.mark.parametrize("case", list(DQN_CASES))
def test_oracle_dqn_family_matches_live_reference_at_wide_obs(case):
    """Three updates (the target network hard-copied after the second) of the oracle from the reference's initialisation against what the reference
    computed"""
    cls, n, d, sharing, seed, bseed, B, kw = DQN_CASES[case]
    g = load_case(LIVE, case)
    it, im = _dqn_index(case)
    n_nets = 1 if sharing else n
    agent_net = [0] * n if sharing else list(range(n))
    torch.manual_seed(seed)   # the reference's initialisation order: agents' networks, their target copies(, mixer)
    theta = lr.init_flat(n_nets, d, A)
    assert np.abs(theta.numpy()[it] - g["theta0"]).max() < 1e-6, "initialisation differs from the reference's"
    hp = lr.DqnHP(**kw)
    if cls == "QMixNetwork":
        lr.init_flat(n_nets, d, A)
        mix = qr.init_mixer_flat(n, n * d, 64, 32)
        assert np.abs(mix.numpy()[im] - g["mix0"]).max() < 1e-6, "mixer initialisation differs from the reference's"
        st = qr.QmixState(theta.clone(), theta.clone(), mix.clone(), mix.clone(), agent_net, d, A)
        update = qr.qmix_update
    else:
        st = lr.DqnState(theta.clone(), theta.clone(), agent_net, d, A)
        update = lr.dqn_update
    rng = np.random.default_rng(bseed)
    for want in g["loss"]:
        got = update(st, _dqn_batch(rng, n, d, B, cls == "QMixNetwork"), hp)
        assert abs(got["loss"] - want) <= 1e-5 * max(1.0, abs(want))
    pairs = [(st.theta, it, "theta"), (st.theta_tgt, it, "theta_tgt")]
    if cls == "QMixNetwork":
        pairs += [(st.mix, im, "mix"), (st.mix_tgt, im, "mix_tgt")]
    for mine, idx, key in pairs:
        assert np.quantile(np.abs(mine.numpy()[idx] - g[key]), 0.999) < 1e-5, key


@pytest.mark.parametrize("case", list(AC_CASES))
def test_oracle_centralised_critic_matches_live_reference_at_wide_obs(case):
    """MAPPO / MAA2C with a 108- / 124-feature centralised critic: the oracle's metrics and parameters after three updates against the reference's"""
    cls, n, d, sharing, seed, bseed, P, steps, kw = AC_CASES[case]
    g = load_case(LIVE, case)
    ia, ic = _ac_index(case)
    assert int(g["critic_in"]) == n * d
    n_nets = 1 if sharing else n
    torch.manual_seed(seed)   # actor drawn before critic, the target critic is a copy
    actor, critic = lr.init_flat(n_nets, d, A), lr.init_flat(n_nets, n * d, 1)
    for mine, key, idx in ((actor, "actor0", ia), (critic, "critic0", ic)):
        assert np.abs(mine.numpy()[idx] - g[key]).max() < 1e-6, f"initialisation differs from the reference's ({key})"
    nets = [0] * n if sharing else list(range(n))
    st = lr.A2CState(actor, critic, critic.clone(), nets, nets, d, A, centralised=True)
    hp = lr.A2CHP(target_update_interval_or_tau=kw["target_update_interval_or_tau"])
    rng = np.random.default_rng(bseed)
    for step, want in zip(steps, g["metrics"]):
        b = _ac_batch(rng, P, n, d)
        got = lr.ppo_update(st, b, hp, step, kw["num_epochs"], kw["ppo_clip"]) if cls == "PPONetwork" else lr.a2c_update(st, b, hp, step)
        np.testing.assert_allclose([got[k] for k in METRICS], want, rtol=1e-5, atol=1e-5)
    for mine, idx, key in ((st.actor, ia, "actor"), (st.critic, ic, "critic"), (st.target, ic, "target")):
        assert np.quantile(np.abs(mine.numpy()[idx] - g[key]), 0.999) < 1e-5, key
