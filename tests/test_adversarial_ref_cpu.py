"""CPU pins of the float64 attack references in adversarial_ref.py (hand-computed cases)."""
import numpy as np

import adversarial_ref as R


def test_linf_step_hand_case():
    x0 = np.array([[0.0, 1.0, -1.0, 2.0]])
    x = np.array([[0.1, 1.2, -1.0, 2.0]])
    g = np.array([[1.0, 3.0, -2.0, 0.0]])
    out = R.step_linf(x, x0, g, [0.25], 0.4)            # a = 0.1
    np.testing.assert_allclose(out, [[0.2, 1.25, -1.1, 2.0]], rtol=0, atol=1e-15)


def test_l2_step_moves_along_g_and_projects():
    x0 = np.zeros((1, 2))
    g = np.array([[3.0, 4.0]])
    # inside the ball: one step of a = 0.5 along g / ||g||
    np.testing.assert_allclose(R.step_l2(x0, x0, g, [1.0], 0.5), [[0.3, 0.4]], atol=1e-15)
    # outside: projected back onto the sphere of radius 1
    out = R.step_l2(np.array([[0.6, 0.8]]), x0, g, [1.0], 0.5)
    np.testing.assert_allclose(out, [[0.6, 0.8]], atol=1e-15)
    out = R.step_l2(np.array([[1.0, 0.0]]), x0, np.array([[0.0, 1.0]]), [1.0], 1.0)
    np.testing.assert_allclose(out, [[2 ** -0.5, 2 ** -0.5]], atol=1e-15)


def test_l2_step_zero_gradient_and_zero_eps():
    x0 = np.array([[1.0, 2.0], [3.0, 4.0]])
    x = x0 + 0.1
    out = R.step_l2(x, x0, np.zeros_like(x0), [1.0, 1.0], 0.5)
    np.testing.assert_array_equal(out, x)
    out = R.step_l2(x, x0, np.ones_like(x0), [0.0, 0.0], 0.5)
    np.testing.assert_array_equal(out, x0)


def test_l2_bound_is_positive_and_grows_with_n():
    rng = np.random.default_rng(0)
    b = [R.l2_step_bound(*(rng.standard_normal((1, n)) for _ in range(3)), [0.5], 0.3).max() for n in (256, 8192)]
    assert 0 < b[0] < b[1] < 1e-3


def test_psr_eps():
    x0 = np.array([[3.0, 4.0, 0.0, 0.0]])                  # ||x0|| = 5, RMS = 2.5
    np.testing.assert_allclose(R.psr_eps(x0, -20.0, "l2"), [0.5])
    np.testing.assert_allclose(R.psr_eps(x0, -20.0, "linf"), [0.25])
    np.testing.assert_allclose(R.psr_eps(x0.reshape(1, 2, 2), 0.0, "l2"), [5.0])
