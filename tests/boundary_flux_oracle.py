"""TEST INFRASTRUCTURE ONLY -- FP64 numpy restatement of the column fluxes with a non-black surface and a warm top
(prb_set_flux_boundaries, then prb_atmosphere_fluxes or prb_atmosphere_band_fluxes).

The fold, levels, integral and non-finite rule of tests/flux_oracle.py and tests/band_flux_oracle.py (the reference's
Layer.transmission along a slant path and its integrateSpectrum), with two other start values:

- top (level L), every node: I = B(nu, t_top); 0 when t_top = 0;
- surface (level 0), node i: I = eps B(nu, t_surface) + (1 - eps) S_i, where eps = 1 gives B exactly.  Lambertian:
  S_i = 2 sum_j w_j mu_j I_down_j(nu, 0), specular: S_i = I_down_i(nu, 0).

eps is np.interp of the table on the Planck axis, rounded to FP32 as the device stores it.  With eps = 1 and t_top = 0
every result equals the existing oracles' bit for bit.
"""
import numpy as np

from oracle import physics as ph
from tests.flux_oracle import FLT_MAX


def emissivity(nu, table):
    """eps(nu) as the device forms it: None -> 1; a scalar -> that constant; (nu_t, eps_t) -> np.interp in FP64.
    Rounded to FP32, returned as FP64."""
    nu = np.asarray(nu, dtype=np.float64)
    if table is None:
        return np.ones_like(nu)
    if np.ndim(table) == 0:
        e = np.full_like(nu, float(table))
    else:
        e = np.interp(nu, np.asarray(table[0], dtype=np.float64), np.asarray(table[1], dtype=np.float64))
    return e.astype(np.float32).astype(np.float64)


def _fold(k, depth_cm, T, t_surface, nu, mu, weights, eps_table, reflection, t_top, add_up, add_down):
    """Both passes per node, downward first; add_up / add_down(j, w, m, I) take every level's radiance.
    Returns (rad_up_top, rad_down_surface), (n_mu, n) each."""
    L = len(depth_cm)
    nu = np.asarray(nu, dtype=np.float64)
    mu, weights = np.atleast_1d(np.asarray(mu, dtype=np.float64)), np.atleast_1d(np.asarray(weights, dtype=np.float64))
    planck = [ph.planck_wavenumber(nu, T[l]) for l in range(L)]
    trans = [[np.exp(-np.asarray(k[l], dtype=np.float64) * depth_cm[l] / m) for l in range(L)] for m in mu]
    rad_down = []
    for i, (m, w) in enumerate(zip(mu, weights)):
        I = ph.planck_wavenumber(nu, t_top) if t_top > 0 else np.zeros_like(nu)
        add_down(L, w, m, I)
        for l in range(L - 1, -1, -1):
            I = ph.transmission(trans[i][l], I, planck[l])
            add_down(l, w, m, I)
        rad_down.append(I)
    eps = emissivity(nu, eps_table)
    b_s = ph.planck_wavenumber(nu, t_surface)
    lamb = sum(2 * w * m * d for m, w, d in zip(mu, weights, rad_down))
    rad_up = []
    for i, (m, w) in enumerate(zip(mu, weights)):
        s = rad_down[i] if reflection == "specular" else lamb
        with np.errstate(invalid="ignore"):
            I = np.where(eps == 1, b_s, eps * b_s + (1 - eps) * s)
        add_up(0, w, m, I)
        for l in range(L):
            I = ph.transmission(trans[i][l], I, planck[l])
            add_up(l + 1, w, m, I)
        rad_up.append(I)
    return np.array(rad_up), np.array(rad_down)


def boundary_fluxes(k, depth_cm, T, t_surface, nu, res, mu, weights, eps_table=None, reflection="lambertian",
                    t_top=0.0):
    """column_fluxes (tests/flux_oracle.py) with the boundaries.  eps_table: None, a scalar or (nu_t, eps_t);
    reflection: "lambertian" or "specular"; t_top in K.  Returns (flux_up, flux_down, rad_up_top, rad_down_surface)."""
    L = len(depth_cm)
    up, down = np.zeros(L + 1), np.zeros(L + 1)

    def adder(flux):
        def add(j, w, m, I):
            flux[j] += 2 * ph.pi * w * m * np.sum(np.where(np.abs(I) <= FLT_MAX, I, 0.0)) * res
        return add

    ru, rd = _fold(k, depth_cm, T, t_surface, nu, mu, weights, eps_table, reflection, t_top, adder(up), adder(down))
    return up, down, ru, rd


def boundary_band_fluxes(k, depth_cm, T, t_surface, nu, res, mu, weights, edges, eps_table=None,
                         reflection="lambertian", t_top=0.0):
    """band_fluxes (tests/band_flux_oracle.py) with the boundaries.  Returns (band_up, band_down), (n_bands, L+1)."""
    L = len(depth_cm)
    nu = np.asarray(nu, dtype=np.float64)
    edges = np.asarray(edges, dtype=np.float64)
    nb = edges.size - 1
    idx = np.searchsorted(edges, nu, side="right") - 1
    sel = (idx >= 0) & (idx < nb)
    up, down = np.zeros((nb, L + 1)), np.zeros((nb, L + 1))

    def adder(flux):
        def add(j, w, m, I):
            I = np.where(np.abs(I) <= FLT_MAX, I, 0.0)
            flux[:, j] += 2 * ph.pi * w * m * np.bincount(idx[sel], weights=I[sel], minlength=nb) * res
        return add

    _fold(k, depth_cm, T, t_surface, nu, mu, weights, eps_table, reflection, t_top, adder(up), adder(down))
    return up, down
