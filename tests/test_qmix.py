"""QMIX (marlbase/dqn/model.py:272-443): the oracle restatement against recorded outputs of the reference and a committed golden vector (CPU), the
CUDA mixer against the oracle (GPU)."""
import os

import numpy as np
import pytest
import torch

from oracle import learner_ref as lr
from oracle import qmix_ref as qr
from tests.helpers import NearTie, load_case, net_layers, redraw_on_near_tie, sample_index

N, T, D, A = 2, 6, 9, 6
GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "qmix_indep.npz")


def _batch(rng, B, n=N, t=T, d=D):
    rew = np.repeat(rng.random((1, t, B)), n, axis=0)
    return dict(obss=torch.tensor(rng.standard_normal((n, t + 1, B, d)), dtype=torch.float32), actions=torch.tensor(rng.integers(0, A, (n, t, B))),
                rewards=torch.tensor(rew, dtype=torch.float32), dones=torch.tensor(rng.random((t + 1, B)) < 0.05, dtype=torch.float32),
                filled=torch.tensor(rng.random((t, B)) < 0.9, dtype=torch.float32))


def _ref_model(ref, ref_shim, tu=2.0, sharing=False):
    return ref.dqn_model.QMixNetwork([ref_shim.Space(shape=(D,))] * N, [ref_shim.Space(n=A)] * N, ref_shim.dqn_cfg(target_update_interval_or_tau=tu), [128, 128],
                                     sharing, False, True, dict(embed_dim=64, hypernet_layers=2, hypernet_embed=32), "cpu")


def _state_from(model, sharing=False):
    kind = "networks" if sharing else "independent"
    n_nets = 1 if sharing else N
    sd = model.state_dict()
    theta = lr.flat_from_state_dict(sd, f"critic.{kind}", n_nets)
    mix = qr.mixer_flat_from_state_dict(sd, "mixer")
    return qr.QmixState(theta.clone(), theta.clone(), mix.clone(), mix.clone(), [0] * N if sharing else list(range(N)), D, A)


LIVE_CASES = [(2.0, False), (0.05, False), (2.0, True)]
LIVE = os.path.join(os.path.dirname(__file__), "golden", "ref_qmix.npz")


def _live_index(sharing):
    return sample_index(net_layers(1 if sharing else N, D, A)), sample_index(qr.mixer_shapes(N, N * D, 64, 32))


def make_reference_cases():
    """Records tests/golden/ref_qmix.npz from the reference's QMixNetwork: MARLBASE_SRC=<marlbase checkout> python -c 'import tests.test_qmix as t;
    t.make_reference_cases()'.  Per case: the loss of each of three updates and the four parameter sets after them at the positions of _live_index."""
    from oracle import ref_shim

    ref = ref_shim.load()
    out = {}
    for c, (tu, sharing) in enumerate(LIVE_CASES):
        torch.manual_seed(11)
        model = _ref_model(ref, ref_shim, tu, sharing)
        kind, n_nets = ("networks", 1) if sharing else ("independent", N)
        it, im = _live_index(sharing)
        sd = model.state_dict()
        out.update({f"c{c}.theta0": lr.flat_from_state_dict(sd, f"critic.{kind}", n_nets).numpy()[it], f"c{c}.mix0": qr.mixer_flat_from_state_dict(sd, "mixer").numpy()[im],
                    f"c{c}.n_mix": np.int64(qr.mixer_flat_from_state_dict(sd, "mixer").numel())})
        rng = np.random.default_rng(5)
        losses = []
        for _ in range(3):
            b = _batch(rng, 16)
            losses.append(model.update(ref.dqn_train.Batch(b["obss"], b["actions"], b["rewards"], b["dones"], b["filled"], None))["loss"])
        sd = model.state_dict()
        out.update({f"c{c}.loss": np.array(losses, np.float64), f"c{c}.theta": lr.flat_from_state_dict(sd, f"critic.{kind}", n_nets).numpy()[it],
                    f"c{c}.theta_tgt": lr.flat_from_state_dict(sd, f"target.{kind}", n_nets).numpy()[it],
                    f"c{c}.mix": qr.mixer_flat_from_state_dict(sd, "mixer").numpy()[im], f"c{c}.mix_tgt": qr.mixer_flat_from_state_dict(sd, "target_mixer").numpy()[im]})
    np.savez_compressed(LIVE, **out)


@pytest.mark.parametrize("tu,sharing", LIVE_CASES)
def test_oracle_matches_live_reference(tu, sharing):
    """Three updates of the oracle against what the reference's QMixNetwork computed from the same initialisation and batches (recorded in
    tests/golden/ref_qmix.npz by make_reference_cases)."""
    g = load_case(LIVE, f"c{LIVE_CASES.index((tu, sharing))}")
    it, im = _live_index(sharing)
    n_nets = 1 if sharing else N
    torch.manual_seed(11)   # the reference's initialisation order: agents' networks, their target copies, mixer
    theta = lr.init_flat(n_nets, D, A)
    lr.init_flat(n_nets, D, A)
    mix = qr.init_mixer_flat(N, N * D, 64, 32)
    assert np.abs(theta.numpy()[it] - g["theta0"]).max() < 1e-6 and np.abs(mix.numpy()[im] - g["mix0"]).max() < 1e-6, "initialisation differs from the reference's"
    st = qr.QmixState(theta.clone(), theta.clone(), mix.clone(), mix.clone(), [0] * N if sharing else list(range(N)), D, A)
    assert st.mix.numel() == qr.mixer_size(N, N * D, 64, 32) == int(g["n_mix"])
    rng = np.random.default_rng(5)
    hp = lr.DqnHP(target_update_interval_or_tau=tu)
    for want in g["loss"]:
        b = _batch(rng, 16)
        got = qr.qmix_update(st, b, hp)
        assert abs(got["loss"] - want) <= 1e-5 * max(1.0, abs(want))
    for mine, idx, key in ((st.theta, it, "theta"), (st.theta_tgt, it, "theta_tgt"), (st.mix, im, "mix"), (st.mix_tgt, im, "mix_tgt")):
        assert np.quantile(np.abs(mine.numpy()[idx] - g[key]), 0.999) < 1e-5, key


def make_golden():
    """Regenerates tests/golden/qmix_indep.npz from the live reference: MARLBASE_SRC=<marlbase checkout> python -c 'import tests.test_qmix as t; t.make_golden()'"""
    from oracle import ref_shim

    ref = ref_shim.load()
    torch.manual_seed(707)
    model = _ref_model(ref, ref_shim, 2.0)
    st = _state_from(model)
    rng = np.random.default_rng(707)
    out = dict(theta0=st.theta.numpy().copy(), mix0=st.mix.numpy().copy())
    for u in range(3):
        b = _batch(rng, 8)
        for k, v in b.items():
            out[f"{k}{u}"] = v.numpy()
        out[f"loss{u}"] = np.float32(model.update(ref.dqn_train.Batch(b["obss"], b["actions"], b["rewards"], b["dones"], b["filled"], None))["loss"])
    sd = model.state_dict()
    out.update(theta3=lr.flat_from_state_dict(sd, "critic.independent", N).numpy(), theta_tgt3=lr.flat_from_state_dict(sd, "target.independent", N).numpy(),
               mix3=qr.mixer_flat_from_state_dict(sd, "mixer").numpy(), mix_tgt3=qr.mixer_flat_from_state_dict(sd, "target_mixer").numpy())
    np.savez_compressed(GOLDEN, **out)


def _golden_batches(g):
    for u in range(3):
        yield {k: torch.tensor(g[f"{k}{u}"]) for k in ("obss", "actions", "rewards", "dones", "filled")}, float(g[f"loss{u}"])


def test_oracle_matches_golden_vector():
    g = np.load(GOLDEN)
    th, mx = torch.tensor(g["theta0"]), torch.tensor(g["mix0"])
    st = qr.QmixState(th.clone(), th.clone(), mx.clone(), mx.clone(), [0, 1], D, A)
    hp = lr.DqnHP(target_update_interval_or_tau=2.0)
    for b, want in _golden_batches(g):
        got = qr.qmix_update(st, b, hp)
        assert abs(got["loss"] - want) <= 1e-5 * max(1.0, abs(want))
    for mine, key in ((st.theta, "theta3"), (st.theta_tgt, "theta_tgt3"), (st.mix, "mix3"), (st.mix_tgt, "mix_tgt3")):
        assert np.quantile(np.abs(mine.numpy() - g[key]), 0.999) < 1e-5, key


@pytest.mark.parametrize("n,s,e,he", [(2, 30, 64, 32), (2, 18, 64, 32), (4, 108, 64, 32), (3, 27, 32, 16), (8, 120, 64, 64), (2, 5, 4, 4), (5, 33, 36, 12)])
def test_weight_gradient_decompositions_cover_every_parameter_exactly_once(n, s, e, he):
    """Host-side invariant of csrc/qmix.cuh (runs without a GPU, through the C ABI): the micro-tiles of the single-read weight-gradient kernel and the
    32 x 32 tiles of the first form each write every mixer parameter exactly once, and the parameter count is the reference's."""
    import ctypes as C

    from codebase_b200 import _native as nat

    lib = nat.lib()
    npar = C.c_int64()
    nat.check(lib.marl_debug_qmix_coverage(C.c_int32(n), C.c_int32(s), C.c_int32(e), C.c_int32(he), None, C.c_int64(0), C.byref(npar)), "marl_debug_qmix_coverage")
    assert npar.value == qr.mixer_size(n, s, e, he)
    counts = (C.c_int32 * (2 * npar.value))()
    nat.check(lib.marl_debug_qmix_coverage(C.c_int32(n), C.c_int32(s), C.c_int32(e), C.c_int32(he), counts, C.c_int64(2 * npar.value), C.byref(npar)), "marl_debug_qmix_coverage")
    c = np.ctypeslib.as_array(counts)
    assert (c[: npar.value] == 1).all(), "single-read form"
    assert (c[npar.value:] == 1).all(), "tile form"


# ---- GPU: the CUDA mixer + the tensor-core training pass of the agents' networks, through the C ABI ---------------------------------------------
def _gpu_model(hp, sharing=False, max_batch=64, n=N, d=D, t=T):
    import types

    from codebase_b200.dqn import model as M

    cfg = types.SimpleNamespace(optimizer="Adam", lr=hp.lr, gamma=hp.gamma, grad_clip=hp.grad_clip, double_q=hp.double_q,
                                target_update_interval_or_tau=hp.target_update_interval_or_tau, standardise_returns=False)
    sp = lambda **kw: types.SimpleNamespace(shape=kw.get("shape"), n=kw.get("n"))
    return M.QMixNetwork([sp(shape=(d,))] * n, [sp(n=A)] * n, cfg, [128, 128], sharing, False, True, dict(embed_dim=64, hypernet_layers=2, hypernet_embed=32), "cuda",
                         max_batch=max_batch, max_episode_length=t)


def _to_store(b, device):
    from codebase_b200.lbf import TrajStore

    n, t1, B, d = b["obss"].shape
    ts = TrajStore(B, n, t1 - 1, d, device)
    ts.obs.copy_(b["obss"].permute(2, 0, 1, 3)); ts.act.copy_(b["actions"].permute(2, 0, 1)); ts.rew.copy_(b["rewards"].permute(2, 0, 1))
    ts.done.copy_(b["dones"].permute(1, 0)); ts.filled.copy_(b["filled"].permute(1, 0))
    return ts


def _scaled_close(got, want, tol, what):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    scale = max(1.0, float(np.abs(want).max()))
    err = float(np.abs(got - want).max())
    assert err <= tol * scale, f"{what}: max abs error {err:.3e} > {tol:g} x {scale:.3g}"


@pytest.mark.gpu
def test_gpu_matches_golden_vector_of_the_reference():
    g = np.load(GOLDEN)
    hp = lr.DqnHP(target_update_interval_or_tau=2.0)
    m = _gpu_model(hp, max_batch=8)
    m.theta.copy_(torch.tensor(g["theta0"])); m.mix.copy_(torch.tensor(g["mix0"]))
    m.params_changed(); m.hard_update()
    for b, want in _golden_batches(g):
        ts = _to_store(b, m.device)
        loss = float(m.update_from_store(ts, torch.arange(8, dtype=torch.int32, device=m.device))[0].item())
        assert abs(loss - want) <= 1e-5 * max(1.0, abs(want))
    for mine, key in ((m.theta, "theta3"), (m.theta_tgt, "theta_tgt3"), (m.mix, "mix3"), (m.mix_tgt, "mix_tgt3")):
        assert np.quantile(np.abs(mine.cpu().numpy() - g[key]), 0.999) < 2e-5, key


@pytest.mark.gpu
@pytest.mark.parametrize("sharing,double_q,tu,B,n,t", [(False, True, 2.0, 16, 2, 6), (True, True, 0.05, 33, 3, 25), (False, False, 200.0, 64, 2, 50), (False, True, 200.0, 5, 4, 7)])
@redraw_on_near_tie
def test_gpu_update_matches_oracle(sharing, double_q, tu, B, n, t):
    hp = lr.DqnHP(double_q=double_q, target_update_interval_or_tau=tu)
    m = _gpu_model(hp, sharing, max_batch=B, n=n, t=t)
    agent_net = [0] * n if sharing else list(range(n))
    # a target that differs from the online networks, so that the double-Q pick and the target mixer matter
    m.theta_tgt.copy_(m.theta + 0.01 * torch.randn_like(m.theta)); m.mix_tgt.copy_(m.mix + 0.01 * torch.randn_like(m.mix)); m.params_changed()
    st = qr.QmixState(m.theta.cpu().clone(), m.theta_tgt.cpu().clone(), m.mix.cpu().clone(), m.mix_tgt.cpu().clone(), agent_net, D, A)
    rng = np.random.default_rng(3)
    for u in range(3):
        b = _batch(rng, B, n=n, t=t)
        if hp.double_q and lr.double_q_margin(lr.DqnState(st.theta, st.theta_tgt, agent_net, D, A), b, hp) < 2e-5:
            raise NearTie()
        st0 = qr.QmixState(st.theta.clone(), st.theta_tgt.clone(), st.mix.clone(), st.mix_tgt.clone(), agent_net, D, A)
        want = qr.qmix_update(st, b, hp)
        ts = _to_store(b, m.device)
        met = m.update_from_store(ts, torch.arange(B, dtype=torch.int32, device=m.device)).cpu()
        filled = float(b["filled"].sum())
        assert abs(float(met[0]) - want["loss"]) <= 1e-5 * max(1.0, abs(want["loss"]))
        got_g = m.grad[: m.n_params].cpu().numpy() / filled
        got_mg = m.mix_grad[: m.n_mix].cpu().numpy() / filled
        _scaled_close(got_mg, want["mix_grad"].numpy(), 2e-5, f"mixer gradient, update {u}")
        err = float(np.abs(got_g - want["grad"].numpy()).max())
        if err > 2e-5 * max(1.0, float(want["grad"].abs().max())):
            if qr.qmix_kink_risk(st0, b, hp) >= 0.5 * err:
                raise NearTie()
            raise AssertionError(f"agents' gradient, update {u}: max abs error {err:.3e}")
        assert abs(float(met[1]) - want["grad_norm"]) <= 2e-5 * max(1.0, want["grad_norm"])
        for mine, theirs, what in ((m.theta, st.theta, "theta"), (m.mix, st.mix, "mixer"), (m.theta_tgt, st.theta_tgt, "target"), (m.mix_tgt, st.mix_tgt, "target mixer")):
            assert np.quantile(np.abs(mine.cpu().numpy() - theirs.numpy()), 0.999) < 2e-5, f"{what} after update {u}"
    m.close()


@pytest.mark.gpu
def test_gpu_update_n_and_state_dict_round_trip():
    """update_n (on-device sampling, the driver's path) keeps the mixer training; the state_dict uses the reference's keys."""
    hp = lr.DqnHP(target_update_interval_or_tau=0.01)
    m = _gpu_model(hp, max_batch=32, t=25)
    rng = np.random.default_rng(9)
    ts = _to_store(_batch(rng, 64, t=25), m.device)
    mix0 = m.mix.clone()
    met = m.update_n(ts, 32, 64, 1234, 0, 5).cpu()
    assert m.updates == 5 and np.isfinite(float(met[0])) and float((m.mix - mix0).abs().max()) > 0 and float((m.mix_tgt - mix0).abs().max()) > 0
    sd = m.state_dict()
    assert sd["mixer.hyper_w_1.2.weight"].shape == (N * 64, 32) and sd["target_mixer.V.2.bias"].shape == (1,) and "critic.independent.1.network.4.bias" in sd
    m2 = _gpu_model(hp, max_batch=32, t=25)
    m2.load_state_dict(sd)
    assert torch.equal(m2.mix, m.mix) and torch.equal(m2.mix_tgt, m.mix_tgt) and torch.equal(m2.theta, m.theta)
    m.close(); m2.close()


@pytest.mark.gpu
def test_gpu_two_learners_of_different_size_coexist():
    """The kernels' shared-memory opt-in is a per-function, process-wide attribute: creating a second, smaller learner must not lower the limit the
    first (4 agents: 2.6x the shared memory) still needs."""
    hp = lr.DqnHP()
    big = _gpu_model(hp, max_batch=8, n=4, t=6)
    small = _gpu_model(hp, max_batch=8, n=2, t=6)
    rng = np.random.default_rng(2)
    for m, n in ((small, 2), (big, 4), (small, 2)):
        ts = _to_store(_batch(rng, 8, n=n, t=6), m.device)
        met = m.update_from_store(ts, torch.arange(8, dtype=torch.int32, device=m.device)).cpu()
        assert np.isfinite(float(met[0])) and float(met[4]) > 0
    big.close(); small.close()
