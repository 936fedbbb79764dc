"""TEST INFRASTRUCTURE ONLY -- FP64 numpy restatement of the layer kernels (prb_atmosphere_layer_kernels).

Two restatements of the same definition.  ``brute_force`` folds the base column with one layer swapped for the current
column's, for every layer, and subtracts the base's band fluxes (the fold of tests/flux_oracle.py: Layer.transmission
along a slant path, integrateSpectrum's non-finite rule).  ``layer_kernels`` is the O(L) formula the device evaluates:
the change at the swapped layer's output times the base transmittance of the layers between it and the boundary.  It
also returns the magnitudes the device's FP32 operations round, for the GPU tests' tolerance.
"""
import numpy as np

from oracle import physics as ph
from tests.flux_oracle import FLT_MAX


def _bands(nu, edges):
    edges = np.asarray(edges, dtype=np.float64)
    idx = np.searchsorted(edges, nu, side="right") - 1
    sel = (idx >= 0) & (idx < edges.size - 1)
    return edges.size - 1, idx, sel


def _finite(x):
    return np.where(np.abs(x) <= FLT_MAX, x, 0.0)


def _band_sum(x, nb, idx, sel):
    return np.bincount(idx[sel], weights=x[sel], minlength=nb)


def boundary_fluxes(k, depth_cm, T, t_surface, nu, res, mu, weights, edges, t_top=0.0):
    """Band fluxes of a column at its two boundaries: (F_up at the top, F_down at the surface), (n_bands,) each.  Upward
    from B(nu, t_surface), downward from B(nu, t_top) (0 when t_top = 0)."""
    L = len(depth_cm)
    nu = np.asarray(nu, dtype=np.float64)
    nb, idx, sel = _bands(nu, edges)
    planck = [ph.planck_wavenumber(nu, T[l]) for l in range(L)]
    up, down = np.zeros(nb), np.zeros(nb)
    for m, w in zip(np.atleast_1d(mu), np.atleast_1d(weights)):
        I = ph.planck_wavenumber(nu, t_surface)
        for l in range(L):
            I = ph.transmission(np.exp(-np.asarray(k[l], dtype=np.float64) * depth_cm[l] / m), I, planck[l])
        up += 2 * ph.pi * w * m * _band_sum(_finite(I), nb, idx, sel) * res
        I = ph.planck_wavenumber(nu, t_top) if t_top > 0 else np.zeros_like(nu)
        for l in range(L - 1, -1, -1):
            I = ph.transmission(np.exp(-np.asarray(k[l], dtype=np.float64) * depth_cm[l] / m), I, planck[l])
        down += 2 * ph.pi * w * m * _band_sum(_finite(I), nb, idx, sel) * res
    return up, down


def brute_force(base, cur, nu, res, mu, weights, edges, t_top=0.0):
    """The kernels by definition.  base, cur: dicts with k (L, n), depth_cm, T, t_surface.  Returns (toa_up, surf_down),
    (n_bands, L+1) each: entry l+1 the change when layer l of the base takes cur's state, entry 0 of toa_up the
    surface temperature's, entry 0 of surf_down 0."""
    L = len(base["depth_cm"])
    args = (nu, res, mu, weights, edges, t_top)
    up0, down0 = boundary_fluxes(base["k"], base["depth_cm"], base["T"], base["t_surface"], *args)
    nb = up0.size
    up, down = np.zeros((nb, L + 1)), np.zeros((nb, L + 1))
    up[:, 0] = boundary_fluxes(base["k"], base["depth_cm"], base["T"], cur["t_surface"], *args)[0] - up0
    for l in range(L):
        k = [cur["k"][m] if m == l else base["k"][m] for m in range(L)]
        d = [cur["depth_cm"][m] if m == l else base["depth_cm"][m] for m in range(L)]
        t = [cur["T"][m] if m == l else base["T"][m] for m in range(L)]
        u, dn = boundary_fluxes(k, d, t, base["t_surface"], *args)
        up[:, l + 1], down[:, l + 1] = u - up0, dn - down0
    return up, down


def planck_difference(nu, t, t_new):
    """B(nu, t_new) - B(nu, t) without cancellation: B (e^(x - x') - 1) / (1 - e^-x'), x = c2 nu / t."""
    with np.errstate(all="ignore"):
        b = ph.planck_wavenumber(nu, t)
        dx = ph.c2 * nu * ((t_new - t) / (t * t_new))
        return b * np.expm1(dx) / -np.expm1(-ph.c2 * nu / t_new)


def transmittance_difference(tau, dtau, m, xp=np):
    """T' - T = exp(-(tau + dtau) / m) - exp(-tau / m) without cancellation: T expm1(-dtau / m) where |dtau| / m < 1/2,
    else the plain difference.  The product form alone is 0 * inf = NaN in an opaque layer (T underflows while
    expm1(-dtau / m) overflows) and would drop a finite node."""
    with np.errstate(all="ignore"):
        x = -dtau / m
        return xp.where(abs(x) < 0.5, xp.exp(-tau / m) * xp.expm1(x), xp.exp(-(tau + dtau) / m) - xp.exp(-tau / m))


def layer_kernels(base, cur, nu, res, mu, weights, edges, t_top=0.0):
    """The O(L) formula (arguments as brute_force).  Per node and point, with T = exp(-k d / mu):
    up:   dI = (1 - T')(B' - B) + (T' - T)(I_up_l - B),  times exp(-(S - S_<=l) / mu)
    down: dI = (1 - T')(B' - B) + (T' - T)(I_down_l+1 - B),  times exp(-S_<l / mu)
    surface: exp(-S / mu)(B(T'_s) - B(T_s)).  T' - T and B' - B are formed without cancellation.
    Returns (toa_up, surf_down, mag_up, mag_down), (n_bands, L+1) each; mag is the sum over points and nodes of
    2 pi w mu res U (|(1 - T') dB| + |T' - T| (|I| + |B|)), the magnitudes an FP32 evaluation rounds."""
    L = len(base["depth_cm"])
    nu = np.asarray(nu, dtype=np.float64)
    nb, idx, sel = _bands(nu, edges)
    kb = [np.asarray(base["k"][l], dtype=np.float64) for l in range(L)]
    kc = [np.asarray(cur["k"][l], dtype=np.float64) for l in range(L)]
    db, dc = base["depth_cm"], cur["depth_cm"]
    tau = [kb[l] * db[l] for l in range(L)]
    dtau = [(kc[l] - kb[l]) * dc[l] + kb[l] * (dc[l] - db[l]) for l in range(L)]   # k'd' - kd
    S = np.sum(tau, axis=0)
    planck = [ph.planck_wavenumber(nu, base["T"][l]) for l in range(L)]
    dplanck = [planck_difference(nu, base["T"][l], cur["T"][l]) if cur["T"][l] != base["T"][l] else np.zeros_like(nu)
               for l in range(L)]
    out = [np.zeros((nb, L + 1)) for _ in range(4)]
    up, down, mag_up, mag_down = out

    def add(dst, mag, j, c, a, w, m):
        with np.errstate(all="ignore"):
            c = np.where(np.isfinite(c) & np.isfinite(a), c, 0.0)
            a = np.where(np.isfinite(a), a, 0.0)
        dst[:, j] += 2 * ph.pi * w * m * _band_sum(c, nb, idx, sel) * res
        mag[:, j] += 2 * ph.pi * w * m * _band_sum(a, nb, idx, sel) * res

    with np.errstate(all="ignore"):
        for m, w in zip(np.atleast_1d(mu), np.atleast_1d(weights)):
            bs = ph.planck_wavenumber(nu, base["t_surface"])
            dbs = planck_difference(nu, base["t_surface"], cur["t_surface"]) \
                if cur["t_surface"] != base["t_surface"] else np.zeros_like(nu)
            u = np.exp(-S / m)
            add(up, mag_up, 0, u * dbs, u * np.abs(dbs), w, m)
            for direction, dst, mag in ((1, up, mag_up), (-1, down, mag_down)):
                if direction == 1:
                    I, order = bs, range(L)
                else:
                    I, order = (ph.planck_wavenumber(nu, t_top) if t_top > 0 else np.zeros_like(nu)), range(L - 1, -1, -1)
                rem = S.copy()
                for l in order:
                    t = np.exp(-tau[l] / m)
                    dt = transmittance_difference(tau[l], dtau[l], m)              # T' - T
                    omt = -np.expm1(-(tau[l] + dtau[l]) / m)                     # 1 - T'
                    di = omt * dplanck[l] + dt * (I - planck[l])
                    rem = rem - tau[l]
                    U = np.exp(-rem / m)
                    add(dst, mag, l + 1, U * di, U * (np.abs(omt * dplanck[l]) + np.abs(dt) * (np.abs(I) + np.abs(planck[l]))),
                        w, m)
                    I = ph.transmission(t, I, planck[l])
    return up, down, mag_up, mag_down
