"""Property tests of the restated oracle (hypothesis; CPU): invariants the reference transition must keep."""
import numpy as np
from hypothesis import example, given, settings, strategies as st

from oracle.env_oracle import OracleEnv, commission_mu, normalise_actions


@settings(max_examples=40, deadline=None)
@given(st.integers(2, 40), st.integers(2, 12), st.integers(0, 2 ** 31 - 1), st.sampled_from([0.0, 0.0025, 0.01]))
@example(A=8, W=2, seed=489224, c=0.0)                          # draws a signed row that sums to 1 at step 4
def test_transition_invariants(A, W, seed, c):
    rs = np.random.RandomState(seed)
    E, S = 5, 3 * W
    env = OracleEnv(E, A, W, 5, commission=c)
    for s in range(S):
        act = rs.standard_normal((E, A)).astype(np.float32)
        act[:, 0] = -np.abs(act[:, 0]) - 0.1                    # a negative entry: softmax branch → the target is a simplex
        # ... unless the row also sums to 1 (trading_env.py:58 keeps such a row as is): move those sums away from 1
        act[:, 0] -= np.where(np.abs(act.sum(1) - 1) < 1e-3, np.float32(1), np.float32(0))
        y = (1 + 0.02 * rs.standard_normal((E, A))).astype(np.float32); y[:, 0] = 1
        v_prev = env.value.copy()
        idx_prev = env.idx.copy()
        r, done = env.step(act, y)
        w = env.hist[np.arange(E), (env.idx - 1) % W]
        assert np.all(w >= 0) and np.allclose(w.sum(1), 1, atol=3e-6)          # drifted weights stay a simplex
        assert np.all(env.value > 0)
        np.testing.assert_array_equal(env.idx, (idx_prev + 1) % W)             # ring pointer (weight_buffer.py:22)
        np.testing.assert_array_equal(env.is_full, np.full(E, int(s + 2 >= W), np.uint8))
        assert not done.any()
        if c == 0:
            np.testing.assert_allclose(r, np.log(env.value / v_prev), rtol=0, atol=3e-6)
        else:
            assert np.all(env.value <= v_prev * (y * normalise_actions(act)).sum(1) * (1 + 1e-6))   # commission only costs


@settings(max_examples=60, deadline=None)
@given(st.integers(2, 64), st.integers(0, 2 ** 31 - 1), st.sampled_from([0.0005, 0.0025, 0.01, 0.05]))
def test_commission_factor_is_a_fixed_point_in_unit_interval(A, seed, c):
    rs = np.random.RandomState(seed)
    w_last = rs.dirichlet(np.ones(A), 8).astype(np.float32)
    w = rs.dirichlet(np.ones(A), 8).astype(np.float32)
    mu = commission_mu(w_last, w, c, max_iter=64)
    assert np.all(mu > 0) and np.all(mu <= 1 + 1e-7)
    c2 = 2 * c - c * c
    resid = (1 - c * w_last[:, 0] - c2 * np.maximum(w_last[:, 1:] - mu[:, None] * w[:, 1:], 0).sum(1)) / (1 - c * w[:, 0]) - mu
    assert np.all(np.abs(resid) < 1e-6)
    same = commission_mu(w, w, c)
    assert np.all(same >= 1 - 1e-6 - 0)                        # no trade → (almost) no cost


def test_weight_channel_layout_transitions():
    """get_all(): zero front padding while filling, raw ring order once full (quirk Q8; weight_buffer.py:32-44)."""
    A, W = 3, 4
    env = OracleEnv(1, A, W, 5)
    seen = []
    for s in range(7):
        act = np.full((1, A), 1.0 / A, np.float32)
        y = np.ones((1, A), np.float32)
        env.step(act, y)
        seen.append(env.weight_channel()[0, 0].copy())
    assert list(seen[0] != 0) == [False, False, True, True]     # 2 rows known: padded at the front
    assert list(seen[1] != 0) == [False, True, True, True]
    assert all((x != 0).all() for x in seen[2:])
    np.testing.assert_array_equal(env.weight_channel()[0], env.hist[0].T)   # full: ring order
