"""Shared helpers for the parity tests."""
import ctypes as C
import os

import numpy as np

from learning_environments_b200._abi import LaneCfg

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def param_index(g):
    """Indices into the parameter vector at which a td_update fixture stores thetas / targets / adam_m / adam_v: all of them,
    or the fixed sample `param_idx` of a fixture that would otherwise exceed 1 MB (oracle/gen_golden.py save_td_update)."""
    return g["param_idx"] if "param_idx" in g.files else slice(None)


def cfg_from_bytes(arr):
    c = LaneCfg()
    raw = np.ascontiguousarray(arr, np.uint8).tobytes()
    assert len(raw) == C.sizeof(LaneCfg), "golden le_lane_cfg size mismatch: regenerate fixtures"
    C.memmove(C.byref(c), raw, len(raw))
    return c


def rel_err(a, b, floor=1e-6):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)) if a.size else 0.0


def sync_prefix(gold_actions, got_actions):
    """Number of leading steps on which two action traces agree."""
    n = min(len(gold_actions), len(got_actions))
    neq = np.nonzero(np.asarray(gold_actions[:n]) != np.asarray(got_actions[:n]))[0]
    return int(neq[0]) if neq.size else n


def assert_params_close(got, want, lr, what=""):
    """Adam moves every parameter by <= lr per step whatever the gradient's magnitude, so ulp-level differences in
    near-zero gradients appear as a small fraction of lr on a few parameters: demand |diff| <= 2% of lr everywhere and
    5e-5 relative (to the parameter scale, floor 1e-2) on >= 99% of the parameters."""
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    d = np.abs(got - want)
    assert d.max() <= 0.02 * lr, "%s: max |diff| %.3g exceeds 2%% of lr=%g" % (what, d.max(), lr)
    rel = d / np.maximum(np.abs(want), 1e-2)
    assert (rel < 5e-5).mean() >= 0.99, "%s: only %.2f%% of the parameters within 5e-5" % (what, 100 * (rel < 5e-5).mean())


def first_divergence(ref, got, n):
    """First training step < n at which two lane traces differ in the action taken or in the episode-end decision
    (done > 0.5), or n when they agree.  `ref` / `got`: objects or dicts with action / done arrays."""
    g = (lambda t, k: t[k]) if isinstance(ref, dict) else getattr
    h = (lambda t, k: t[k]) if isinstance(got, dict) else getattr
    a = np.asarray(g(ref, "action")[:n]) != np.asarray(h(got, "action")[:n])
    d = (np.asarray(g(ref, "done")[:n]) > 0.5) != (np.asarray(h(got, "done")[:n]) > 0.5)
    bad = np.nonzero(a | d)[0]
    return int(bad[0]) if bad.size else n


def assert_divergence_is_near_tie(ref, got, t, what=""):
    """A lane may leave the reference trajectory only at a near-tie (BASELINE north_star: "argmax actions bit-exact away from
    stated near-ties").  Up to step t both sides took identical actions on identical Philox draws, so their Q-values differ
    only by accumulated rounding; a different greedy action (or a different done > 0.5 decision on the SE's real-valued
    done output) then means the two candidates were closer than that rounding.  The admissible relative gap is
    max(1e-5, 10 x drift), drift = the largest relative deviation of the TD losses / next states over the common prefix —
    the rounding drift this very lane has accumulated, measured, not assumed.  `ref` may lack qgap (reference goldens)."""
    g = (lambda tr, k: tr[k]) if isinstance(ref, dict) else getattr
    h = (lambda tr, k: tr[k]) if isinstance(got, dict) else getattr
    assert np.array_equal(np.asarray(g(ref, "explore")[:t + 1]), np.asarray(h(got, "explore")[:t + 1])), what + ": explore flags are Philox-exact"
    lr, lg = np.asarray(g(ref, "loss")[:t], np.float64), np.asarray(h(got, "loss")[:t], np.float64)
    k = ~np.isnan(lr) & ~np.isnan(lg)
    drift = float(np.max(np.abs(lr[k] - lg[k]) / np.maximum(np.abs(lr[k]), 1e-6))) if k.any() else 0.0
    sr, sg = np.asarray(g(ref, "next_state")[:t], np.float64), np.asarray(h(got, "next_state")[:t], np.float64)
    if t > 0:
        drift = max(drift, float(np.max(np.abs(sr - sg) / np.maximum(np.abs(sr), 1e-2))))
    tol = max(1e-5, 10.0 * drift)
    if int(g(ref, "action")[t]) != int(h(got, "action")[t]):
        assert not int(h(got, "explore")[t]), what + ": random actions are Philox-exact, a difference there is a bug"
        gaps = [abs(float(h(got, "qgap")[t]))]
        try:
            gaps.append(abs(float(g(ref, "qgap")[t])))
        except (KeyError, AttributeError, IndexError, TypeError):
            pass
        gap = np.nanmin(gaps)
        assert gap <= tol, "%s: left the reference at step %d with a relative Q gap of %.3g (> %.3g = near-tie bound from a drift of %.3g)" % (
            what, t, gap, tol, drift)
    else:   # same action, different episode-end decision: the SE's done output sat at the 0.5 threshold
        dr, dg = float(g(ref, "done")[t]), float(h(got, "done")[t])
        assert min(abs(dr - 0.5), abs(dg - 0.5)) <= tol * max(1.0, abs(dr)), "%s: done threshold decision differs at step %d (%.6g vs %.6g)" % (what, t, dr, dg)
    return tol
