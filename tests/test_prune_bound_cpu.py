"""The bound that lets EI-CF / PI-CF sweeps skip candidates (acq.cu: prune_bound_kernel), restated in numpy and checked
against brute force on near-boundary cases: f* placed a few ulps above and below the largest utility the sweep's
arithmetic can produce.  A candidate the bound prunes must never have a base sample with U > f*; a candidate with
such a sample must always survive, and so must one with a NaN anywhere."""
import numpy as np
import pytest

U_RND = 2.0 ** -53
COMPOSITES = ("sumsq_target", "rosen_composite", "neg_sum_exp", "linear")


def sd_max(variance, noise):
    """smax_j of the kernel: sqrt(max(sigma_f^2 + noise, 1e-10)), inflated by 2^-47."""
    return np.sqrt(np.maximum(variance + noise, 1e-10)) * (1.0 + 2.0 ** -47)


def _seg_max(composite, th, lo, hi):
    """(bound, magnitude) of phi_j over [lo, hi] per output; th: theta_j (sumsq / linear) or a (rosen)."""
    m = lo.shape[-1]
    if composite in ("sumsq_target", "rosen_composite"):
        tgt = np.broadcast_to(th, lo.shape)
        if composite == "rosen_composite":
            j = np.arange(m)
            tgt = np.where(j < m // 2, th[..., :1] if np.ndim(th) else th, 0.0) * np.ones_like(lo)
        d1, d2 = lo - tgt, tgt - hi
        dist = np.where(~(d1 <= 0), d1, np.where(~(d2 <= 0), d2, 0.0))       # a NaN propagates
        b = -(dist * dist)
        if composite == "rosen_composite":
            j = np.arange(m)
            b = np.where(j < m // 2, b, np.where(j < 2 * (m // 2), -(100.0 * (dist * dist)), 0.0))
        return b, -b
    if composite == "neg_sum_exp":
        b = -np.exp(lo)
        return b, -b
    b = th * np.where(th >= 0, hi, lo)
    return b, np.abs(th) * np.maximum(np.abs(lo), np.abs(hi))


def bound_plus_margin(composite, mu, smax, Z, theta):
    """(N, S): sum_j segment maximum + margin per candidate mu (N, m) and base sample Z (S, m), with smax (m,) and theta
    (m,) ((1,) for rosen), formed as the kernel forms it."""
    m = mu.shape[1]
    e = mu[:, None, :] + smax[None, None, :] * Z[None, :, :]          # two roundings, as the kernel (no contraction)
    up = Z[None, :, :] >= 0
    lo, hi = np.where(up, mu[:, None, :], e), np.where(up, e, mu[:, None, :])
    b, mag = _seg_max(composite, theta, lo, hi)
    ub = np.zeros(b.shape[:2])
    mg = np.zeros(b.shape[:2])
    for j in range(m):                                              # sequential sums, as the kernel
        ub = ub + b[..., j]
        mg = mg + mag[..., j]
    cm = (4.0 * m + 16.0) * U_RND
    return ub + (cm * mg + 1e-300)


def survives(composite, mu, smax, Z, theta, fstar):
    """The kernel's decision: True unless bound + margin <= f* for every sample."""
    return np.any(~(bound_plus_margin(composite, mu, smax, Z, theta) <= np.reshape(fstar, (-1, 1))), axis=1)


def sweep_utility(composite, mu, sigma, Z, theta, fma):
    """U_s of mc_acq_kernel at candidates mu (N, m) with sigma (N, m): y = mu + sigma z with one rounding (fma, emulated in
    extended precision) or two, then phi summed over outputs in order."""
    if fma:
        y = (mu[:, None, :].astype(np.longdouble) + sigma[:, None, :].astype(np.longdouble) * Z[None].astype(np.longdouble)).astype(np.float64)
    else:
        y = mu[:, None, :] + sigma[:, None, :] * Z[None]
    m = mu.shape[1]
    if composite == "sumsq_target":
        t = -((y - theta) * (y - theta))
    elif composite == "rosen_composite":
        j = np.arange(m)
        t = np.where(j < m // 2, -((theta[0] - y) * (theta[0] - y)), np.where(j < 2 * (m // 2), -(100.0 * (y * y)), 0.0))
    elif composite == "neg_sum_exp":
        t = -np.exp(y)
    else:
        t = theta * y
    U = np.zeros(y.shape[:2])
    for j in range(m):
        U = U + t[..., j]
    return U


def _case(composite, seed, N=400, m=6, S=64):
    rng = np.random.default_rng(seed)
    mu = rng.normal(0.0, 1.0, size=(N, m)) * rng.choice([1e-3, 1.0, 30.0], size=(N, 1))
    var_f = rng.uniform(0.5, 2.0, size=m)
    noise = rng.choice([0.0, 1e-6, 1e-2], size=m)
    Z = rng.standard_normal((S, m))
    theta = rng.normal(size=m) if composite != "rosen_composite" else np.array([rng.uniform(0.5, 1.5)])
    if composite == "linear":
        theta = rng.dirichlet(np.ones(m)) * rng.choice([-1.0, 1.0], size=m)
    # the sweep's sigma: at the prior maximum (the far end of every segment) or anywhere below it
    smax0 = np.sqrt(np.maximum(var_f + noise, 1e-10))
    frac = np.where(rng.uniform(size=(N, 1)) < 0.5, 1.0, rng.uniform(size=(N, m)))
    sigma = np.sqrt(np.maximum(noise + var_f * frac, 1e-10))
    sigma = np.minimum(sigma, smax0)
    return mu, sd_max(var_f, noise), sigma, Z, theta


@pytest.mark.parametrize("composite", COMPOSITES)
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_bound_never_prunes_an_active_candidate(composite, seed):
    mu, smax, sigma, Z, theta = _case(composite, seed)
    for fma in (False, True):
        Umax = sweep_utility(composite, mu, sigma, Z, theta, fma).max(axis=1)
        for k in range(-4, 5):
            # f* a few ulps around the candidate's largest utility: active where Umax > f*
            fstar = np.nextafter(Umax, np.inf * np.sign(k)) if k else Umax
            for _ in range(abs(k) - 1):
                fstar = np.nextafter(fstar, np.inf * np.sign(k))
            keep = np.array([survives(composite, mu[i:i + 1], smax, Z, theta, fstar[i])[0] for i in range(len(mu))])
            assert np.all(keep[Umax > fstar])


@pytest.mark.parametrize("composite", COMPOSITES)
def test_bound_prunes_far_candidates(composite):
    """The bound is not vacuous: with f* just above the largest segment maximum plus the margin, everything is pruned,
    and with f* a few ulps below the sweep's largest utility, everything survives."""
    mu, smax, sigma, Z, theta = _case(composite, 7, N=100)
    cut = bound_plus_margin(composite, mu, smax, Z, theta).max(axis=1)
    assert not np.any([survives(composite, mu[i:i + 1], smax, Z, theta, np.nextafter(cut[i], np.inf))[0]
                       for i in range(len(mu))])
    Umax = sweep_utility(composite, mu, sigma, Z, theta, False).max(axis=1)
    below = np.nextafter(np.nextafter(Umax, -np.inf), -np.inf)
    assert np.all([survives(composite, mu[i:i + 1], smax, Z, theta, below[i])[0] for i in range(len(mu))])


def test_margin_covers_rounding_at_the_boundary():
    """sumsq_target with the sweep's sigma at the prior maximum and the target on a segment's far end: the utility the
    sweep computes can exceed the exactly rounded bound by a few ulps, and the margin keeps such candidates."""
    rng = np.random.default_rng(3)
    m, S = 16, 32
    Z = rng.standard_normal((S, m))
    var_f, noise = np.ones(m), np.full(m, 1e-2)
    smax0 = np.sqrt(var_f + noise)
    mu = rng.normal(size=(200, m))
    theta = mu[0] + smax0 * Z[0] * (1.0 - 1e-15)                     # the first candidate's sample 0 hits the target
    for fma in (False, True):
        U = sweep_utility("sumsq_target", mu, np.tile(smax0, (200, 1)), Z, theta, fma)
        Umax = U.max(axis=1)
        fstar = np.nextafter(Umax, -np.inf)
        keep = survives("sumsq_target", mu, sd_max(var_f, noise), Z, theta, fstar)
        assert np.all(keep)


@pytest.mark.parametrize("where", ["mu", "theta", "fstar", "z"])
def test_nan_survives(where):
    mu, smax, sigma, Z, theta = _case("sumsq_target", 4, N=5)
    fstar = 1e300
    if where == "mu":
        mu[2, 1] = np.nan
    elif where == "theta":
        theta = theta.copy()
        theta[0] = np.nan
    elif where == "fstar":
        fstar = np.nan
    else:
        Z = Z.copy()
        Z[3, 0] = np.nan
    keep = survives("sumsq_target", mu, smax, Z, theta, fstar)
    assert keep[2] if where == "mu" else np.all(keep)
