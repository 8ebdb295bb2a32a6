"""Shared helpers of the GPU parity tests."""
import functools

import pytest
import torch

TIE = 2e-5   # relative gap of the two best online Q-values under which the double-Q argmax may legitimately differ between two implementations


class NearTie(Exception):
    """The seeded case sits on a discontinuity of the loss gradient -- a double-Q argmax margin below TIE, or a ReLU unit at its kink with a visible
    gradient share: comparing against the oracle would be a coin toss."""


def check_margin(lr, st, batch, hp):
    if lr.double_q_margin(st, batch, hp) < TIE:
        raise NearTie()


def assert_grad_close(lr, st, batch, hp, got, want, tol=1e-5, what=""):
    """max |got - want| <= tol x max(1, max |want|).  A mismatch that a single ReLU unit sitting on its kink explains is a NearTie, not a failure: a
    hidden pre-activation within ~1e-6 of zero may be "on" in one implementation and "off" in the other (they agree to ~5e-7), which moves the
    gradient by up to dL/dh x (the unit's input row) = oracle.learner_ref.dqn_kink_risk -- e.g. 1.3e-3 for VDN at batch 16, T = 127, where the
    defect-free kernels of two consecutive builds "failed" this way.  The excuse only covers mismatches up to twice that bound."""
    import numpy as np

    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    scale = max(1.0, float(np.abs(want).max()))
    err = float(np.abs(got - want).max())
    if err <= tol * scale:
        return
    risk = lr.dqn_kink_risk(st, batch, hp)
    if risk >= 0.5 * err:
        raise NearTie()
    raise AssertionError(f"{what} max abs error {err:.3e} > {tol:g} x {scale:.3g} (largest ReLU-kink move of this case: {risk:.3e})")


def net_layers(n_nets, in_dim, out_dim, hidden=128):
    """(out, in) of every Linear layer of `n_nets` FCNetworks, in the order of the flat parameter vector."""
    return [(hidden, in_dim), (hidden, hidden), (out_dim, hidden)] * n_nets


def sample_index(layers, per_tensor=64):
    """Positions at which the recorded reference outputs (tests/golden/ref_*.npz) keep a flat parameter vector made of consecutive Linear layers
    (weight, then bias): at most `per_tensor` evenly spaced elements of every weight and every bias, so that each tensor is checked while the files
    stay small."""
    import numpy as np

    out, o = [], 0
    for no, ni in layers:
        for n in (no * ni, no):
            out.append(o + np.unique(np.linspace(0, n - 1, min(n, per_tensor)).round().astype(np.int64)))
            o += n
    return np.concatenate(out)


def load_case(path, case):
    """The arrays of one recorded case (keys `<case>.<name>`) of a tests/golden/ref_*.npz file."""
    import numpy as np

    with np.load(path) as g:
        return {k[len(case) + 1:]: g[k] for k in g.files if k.startswith(case + ".")}


def redraw_on_near_tie(fn):
    """Run the test body with seeds 0, 1, ... until its oracle argmax margin is healthy (at most five draws): with a healthy margin every mismatch
    is a defect; five near-ties in a row are not plausible (they occur in ~8 % of random initialisations, tools/grad_stress.py)."""

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        for attempt in range(5):
            torch.manual_seed(7919 * attempt + 17)
            try:
                return fn(*args, **kwargs)
            except NearTie:
                continue
        pytest.fail("five initialisations in a row hit a double-Q near-tie: not plausible")

    return wrapper
