"""cfg.standardise_returns of the DQN family (marlbase/dqn/model.py:82-84,147-158; VDN 221-222,256-264): the oracle against recorded outputs of the
reference classes (tests/golden/ref_standardise_returns_dqn.npz) and the B200 path (marl_dqn_standardise_returns) against the oracle."""
import copy
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


def _store(rng, cap, coop):
    obs = rng.integers(-1, 8, size=(cap, N, T + 1, D)).astype(np.float32)
    act = rng.integers(0, A, size=(cap, N, T)).astype(np.int32)
    rew = 3.0 * (rng.random((cap, N, T)) < 0.3).astype(np.float32) * rng.random((cap, N, T)).astype(np.float32)
    if coop:
        rew[:] = rew[:, :1]
    length = rng.integers(1, T + 1, size=cap)
    done = np.zeros((cap, T + 1), np.uint8); filled = np.zeros((cap, T), np.uint8)
    for e in range(cap):
        filled[e, : length[e]] = 1
        done[e, length[e]] = rng.random() < 0.7
    return dict(obs=obs, act=act, rew=rew, done=done, filled=filled)


LIVE = os.path.join(os.path.dirname(__file__), "golden", "ref_standardise_returns_dqn.npz")


def _live_batches(mixer, B=12):
    rng = np.random.default_rng(8)
    for _ in range(3):
        s = _store(rng, 40, bool(mixer))
        yield lr.batch_from_store(s, rng.integers(0, 40, size=B).astype(np.int32))


def make_reference_cases():
    """Records tests/golden/ref_standardise_returns_dqn.npz from the reference's QNetwork / VDNetwork: MARLBASE_SRC=<marlbase checkout> python -c
    'import tests.test_standardise_returns_dqn as t; t.make_reference_cases()'."""
    from oracle import ref_shim

    ref = ref_shim.load()
    idx = sample_index(net_layers(N, D, A))
    out = {}
    for cls in ("QNetwork", "VDNetwork"):
        torch.manual_seed(3)
        model = getattr(ref.dqn_model, cls)([ref_shim.Space(shape=(D,))] * N, [ref_shim.Space(n=A)] * N, ref_shim.dqn_cfg(standardise_returns=True), [128, 128], False, False, True, "cpu")
        out[f"{cls}.theta0"] = lr.flat_from_state_dict(model.state_dict(), "critic.independent", N).numpy()[idx]
        losses = [model.update(ref.dqn_train.Batch(b["obss"], b["actions"], b["rewards"], b["dones"], b["filled"], None))["loss"]
                  for b in _live_batches(int(cls == "VDNetwork"))]
        out.update({f"{cls}.loss": np.array(losses, np.float64), f"{cls}.ret_mean": model.ret_ms.mean.numpy(), f"{cls}.ret_var": model.ret_ms.var.numpy(),
                    f"{cls}.theta": lr.flat_from_state_dict(model.state_dict(), "critic.independent", N).numpy()[idx]})
    np.savez_compressed(LIVE, **out)


@pytest.mark.parametrize("cls,mixer", [("QNetwork", 0), ("VDNetwork", 1)])
def test_oracle_matches_live_reference(cls, mixer):
    """Three updates of the oracle against what the reference's class computed from the same initialisation and batches (recorded by
    make_reference_cases)."""
    g = load_case(LIVE, cls)
    idx = sample_index(net_layers(N, D, A))
    torch.manual_seed(3)
    theta = lr.init_flat(N, D, A)
    assert np.abs(theta.numpy()[idx] - g["theta0"]).max() < 1e-6, "initialisation differs from the reference's"
    st = lr.DqnState(theta.clone(), theta.clone(), [0, 1], D, A, ret_ms=lr.RunningMeanStdRef((1,) if mixer else (N,)))
    hp = lr.DqnHP(mixer=mixer)
    for b, want in zip(_live_batches(mixer), g["loss"], strict=True):
        _close(lr.dqn_update(st, b, hp)["loss"], want)
    _close(st.ret_ms.mean.numpy(), g["ret_mean"]); _close(st.ret_ms.var.numpy(), g["ret_var"])
    d = np.abs(st.theta.numpy()[idx] - g["theta"])
    assert np.quantile(d, 0.999) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("mixer,B,sharing", [(0, 64, False), (0, 700, True), (1, 48, False), (1, 257, False)])
def test_device_matches_oracle(mixer, B, sharing):
    from codebase_b200.dqn import model as M
    from codebase_b200.lbf import TrajStore

    rng = np.random.default_rng(B)
    hp = lr.DqnHP(mixer=mixer, target_update_interval_or_tau=2)
    cfg = types.SimpleNamespace(optimizer="Adam", lr=hp.lr, gamma=hp.gamma, grad_clip=hp.grad_clip, double_q=True, target_update_interval_or_tau=2, standardise_returns=True)
    m = (M.VDNetwork if mixer else M.QNetwork)([_space(shape=(D,))] * N, [_space(n=A)] * N, cfg, [128, 128], sharing, False, True, "cuda", max_batch=B, max_episode_length=T)
    st = lr.DqnState(m.theta.cpu().clone(), m.theta_tgt.cpu().clone(), m.agent_net, D, A, ret_ms=lr.RunningMeanStdRef((1,) if mixer else (N,)))
    for u in range(3):
        s = _store(rng, 300, bool(mixer))
        idx = rng.integers(0, 300, size=B).astype(np.int32)
        batch = lr.batch_from_store(s, idx)
        if lr.double_q_margin(st, batch, hp) < 2e-5:
            pytest.skip("double-Q near-tie in this draw")
        want = lr.dqn_update(st, batch, hp)
        ts = TrajStore(300, N, T, D, m.device)
        for k in ("obs", "act", "rew", "done", "filled"):
            getattr(ts, k).copy_(torch.as_tensor(s[k]))
        m.update_grads(ts, torch.tensor(idx, device="cuda"))
        gr = m.grad.cpu().numpy(); n = m.n_params
        scale = max(1.0, float(np.abs(want["grad"].numpy()).max()))
        _close(gr[:n] / gr[n + 1] / scale, want["grad"].numpy() / scale, rtol=2e-5, atol=2e-5)
        _close(m.update_apply().cpu().numpy()[0], want["loss"], rtol=2e-5, atol=2e-5)
        mean, var, count = m.ret_ms()
        ref_mean = st.ret_ms.mean.numpy() if st.ret_ms.mean.numel() > 1 else np.full(len(mean), float(st.ret_ms.mean))
        _close(mean.numpy(), ref_mean); _close(var.numpy(), st.ret_ms.var.numpy() if st.ret_ms.var.numel() > 1 else np.full(len(var), float(st.ret_ms.var)))
        assert abs(count - st.ret_ms.count) < 1e-6
        m.theta.copy_(st.theta); m.theta_tgt.copy_(st.theta_tgt); m.adam_m.copy_(st.m); m.adam_v.copy_(st.v)
        m.params_changed()
