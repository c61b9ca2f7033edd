"""float64 references of the projected-gradient attack step (amc_adv_step) and of the PSR budget of PGDAttack
(tests/test_gpu_adversarial.py), pinned on the CPU by tests/test_adversarial_ref_cpu.py.  Frames are rows of [B, n]."""
import numpy as np


def step_linf(x, x0, g, eps, step_frac):
    """x = min(max(x + a sign(g), x0 - eps), x0 + eps), a = step_frac * eps, per frame."""
    x, x0, g = (np.asarray(t, np.float64) for t in (x, x0, g))
    e = np.asarray(eps, np.float64)[:, None]
    return np.minimum(np.maximum(x + step_frac * e * np.sign(g), x0 - e), x0 + e)


def step_l2(x, x0, g, eps, step_frac):
    """v = x + a g / ||g|| (v = x when ||g|| = 0); d = v - x0; x = ||d|| > eps ? x0 + d eps / ||d|| : v."""
    x, x0, g = (np.asarray(t, np.float64) for t in (x, x0, g))
    e = np.asarray(eps, np.float64)[:, None]
    gn = np.linalg.norm(g, axis=1, keepdims=True)
    v = x + np.where(gn > 0, step_frac * e / np.where(gn > 0, gn, 1.0), 0.0) * g
    d = v - x0
    dn = np.linalg.norm(d, axis=1, keepdims=True)
    return np.where(dn > e, x0 + d * (e / np.where(dn > 0, dn, 1.0)), v)


def l2_step_bound(x, x0, g, eps, step_frac):
    """Per-element bound on |fp32 kernel - step_l2| from the kernel's fp32 arithmetic (unit roundoff u = 2^-24).

    Each of the two frame norms is a sum of squares accumulated sequentially per thread (ceil(n / 256) terms), then over
    5 warp-shuffle levels and 8 warp partials, and a square root: relative error <= (ceil(n/256) + 14) u.  The step
    scale a / ||g|| and the projection ratio eps / ||d|| each add two roundings, and the element-wise update, difference
    and projection add one rounding each of the magnitudes involved.  The factor 4 covers the propagation of the norm
    errors through both scales and the final add."""
    x, x0, g = (np.asarray(t, np.float64) for t in (x, x0, g))
    n = x.shape[1]
    u = 2.0 ** -24
    k = 4.0 * (np.ceil(n / 256.0) + 14.0 + 4.0)
    e = np.asarray(eps, np.float64)[:, None]
    gn = np.linalg.norm(g, axis=1, keepdims=True)
    ag = np.where(gn > 0, step_frac * e * np.abs(g) / np.where(gn > 0, gn, 1.0), 0.0)
    d = np.abs(x + ag - x0) + ag
    return k * u * (np.abs(x0) + np.abs(x) + ag + d)


def psr_eps(x0, psr_db, norm):
    """Per-frame budget for a perturbation-to-signal ratio in dB: L2 10^(psr/20) ||x0_b||, L-inf that over sqrt(n)."""
    x0 = np.asarray(x0, np.float64).reshape(len(x0), -1)
    e = 10.0 ** (psr_db / 20.0) * np.linalg.norm(x0, axis=1)
    return e / np.sqrt(x0.shape[1]) if norm == "linf" else e
