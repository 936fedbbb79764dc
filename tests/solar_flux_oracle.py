"""TEST INFRASTRUCTURE ONLY -- FP64 numpy restatement of the column fluxes with a solar beam (prb_set_solar_source, with
or without prb_set_flux_boundaries, then prb_atmosphere_fluxes or prb_atmosphere_band_fluxes).

The fold, levels, integral, boundaries and non-finite rule of tests/boundary_flux_oracle.py, plus a collimated beam along
mu_sun that is absorbed and neither emitted into nor scattered:

- E(nu, L) = S(nu), E <- E exp(-k_l depth_l / mu_sun) through layer l going down; flux_down[j] gains
  mu_sun sum E(nu, j) res;
- the surface reflects 1 - eps of E(nu, 0) (eps = 1 reflects exactly nothing).  Lambertian: every node's upward start
  is eps B + (1 - eps) (S_i + mu_sun E(nu, 0) / pi).  Specular: a beam E_up = (1 - eps) E(nu, 0) rises along mu_sun
  through the same layer factors, and flux_up[j] gains mu_sun sum E_up(nu, j) res.

S is np.interp(nu, nu_t, S_t, left=0, right=0), rounded to FP32 as the device stores it; eps is the boundary oracle's.
With S = 0 every result equals the boundary oracle's bit for bit.
"""
import numpy as np

from oracle import physics as ph
from tests.boundary_flux_oracle import emissivity
from tests.flux_oracle import FLT_MAX


def irradiance(nu, table):
    """S(nu) as the device forms it: None -> 0; (nu_t, S_t) -> np.interp in FP64 with 0 outside the table, rounded to
    FP32.  Returned as FP64."""
    nu = np.asarray(nu, dtype=np.float64)
    if table is None:
        return np.zeros_like(nu)
    s = np.interp(nu, np.asarray(table[0], dtype=np.float64), np.asarray(table[1], dtype=np.float64), left=0, right=0)
    return s.astype(np.float32).astype(np.float64)


def solar_beam(k, depth_cm, nu, sun, mu_sun):
    """The downward beam at every level: (L+1, n), row j = E(nu, level j); row L = S, row 0 reaches the surface."""
    L = len(depth_cm)
    e = np.empty((L + 1, np.asarray(nu).size))
    e[L] = irradiance(nu, sun)
    for l in range(L - 1, -1, -1):
        e[l] = e[l + 1] * np.exp(-np.asarray(k[l], dtype=np.float64) * depth_cm[l] / mu_sun)
    return e


def _masked(I):
    return np.where(np.abs(I) <= FLT_MAX, I, 0.0)


def _fold(k, depth_cm, T, t_surface, nu, mu, weights, eps_table, reflection, t_top, sun, mu_sun, add_up, add_down):
    """Both passes, downward first; add_up / add_down(j, c, I) add c sum I res at level j (c = 2 pi w mu for a node,
    mu_sun for a beam).  Returns (rad_up_top, rad_down_surface), (n_mu, n) each."""
    L = len(depth_cm)
    nu = np.asarray(nu, dtype=np.float64)
    mu, weights = np.atleast_1d(np.asarray(mu, dtype=np.float64)), np.atleast_1d(np.asarray(weights, dtype=np.float64))
    planck = [ph.planck_wavenumber(nu, T[l]) for l in range(L)]
    trans = [[np.exp(-np.asarray(k[l], dtype=np.float64) * depth_cm[l] / m) for l in range(L)] for m in mu]
    rad_down = []
    for i, (m, w) in enumerate(zip(mu, weights)):
        I = ph.planck_wavenumber(nu, t_top) if t_top > 0 else np.zeros_like(nu)
        add_down(L, 2 * ph.pi * w * m, I)
        for l in range(L - 1, -1, -1):
            I = ph.transmission(trans[i][l], I, planck[l])
            add_down(l, 2 * ph.pi * w * m, I)
        rad_down.append(I)
    beam = solar_beam(k, depth_cm, nu, sun, mu_sun)
    for j in range(L, -1, -1):
        add_down(j, mu_sun, beam[j])
    eps = emissivity(nu, eps_table)
    b_s = ph.planck_wavenumber(nu, t_surface)
    lamb = sum(2 * w * m * d for m, w, d in zip(mu, weights, rad_down)) + mu_sun * beam[0] / ph.pi
    rad_up = []
    for i, (m, w) in enumerate(zip(mu, weights)):
        s = rad_down[i] if reflection == "specular" else lamb
        with np.errstate(invalid="ignore"):
            I = np.where(eps == 1, b_s, eps * b_s + (1 - eps) * s)
        add_up(0, 2 * ph.pi * w * m, I)
        for l in range(L):
            I = ph.transmission(trans[i][l], I, planck[l])
            add_up(l + 1, 2 * ph.pi * w * m, I)
        rad_up.append(I)
    if reflection == "specular":
        e = np.where(eps == 1, 0.0, (1 - eps) * beam[0])
        add_up(0, mu_sun, e)
        for l in range(L):
            e = e * np.exp(-np.asarray(k[l], dtype=np.float64) * depth_cm[l] / mu_sun)
            add_up(l + 1, mu_sun, e)
    return np.array(rad_up), np.array(rad_down)


def solar_fluxes(k, depth_cm, T, t_surface, nu, res, mu, weights, sun=None, mu_sun=1.0, eps_table=None,
                 reflection="lambertian", t_top=0.0):
    """boundary_fluxes (tests/boundary_flux_oracle.py) with the Sun.  sun: None or (nu_t, S_t) in W m-2 (cm-1)-1;
    mu_sun in (0, 1].  Returns (flux_up, flux_down, rad_up_top, rad_down_surface)."""
    L = len(depth_cm)
    up, down = np.zeros(L + 1), np.zeros(L + 1)

    def adder(flux):
        def add(j, c, I):
            flux[j] += c * np.sum(_masked(I)) * res
        return add

    ru, rd = _fold(k, depth_cm, T, t_surface, nu, mu, weights, eps_table, reflection, t_top, sun, mu_sun, adder(up),
                   adder(down))
    return up, down, ru, rd


def solar_band_fluxes(k, depth_cm, T, t_surface, nu, res, mu, weights, edges, sun=None, mu_sun=1.0, eps_table=None,
                      reflection="lambertian", t_top=0.0):
    """boundary_band_fluxes (tests/boundary_flux_oracle.py) with the Sun.  Returns (band_up, band_down),
    (n_bands, L+1) each."""
    L = len(depth_cm)
    nu = np.asarray(nu, dtype=np.float64)
    edges = np.asarray(edges, dtype=np.float64)
    nb = edges.size - 1
    idx = np.searchsorted(edges, nu, side="right") - 1
    sel = (idx >= 0) & (idx < nb)
    up, down = np.zeros((nb, L + 1)), np.zeros((nb, L + 1))

    def adder(flux):
        def add(j, c, I):
            flux[:, j] += c * np.bincount(idx[sel], weights=_masked(I)[sel], minlength=nb) * res
        return add

    _fold(k, depth_cm, T, t_surface, nu, mu, weights, eps_table, reflection, t_top, sun, mu_sun, adder(up), adder(down))
    return up, down


def beam_flux_down(k, depth_cm, nu, res, sun, mu_sun):
    """The beam's share of flux_down at every level: mu_sun sum E(nu, j) res, (L+1,)."""
    return np.array([mu_sun * np.sum(_masked(e)) * res for e in solar_beam(k, depth_cm, nu, sun, mu_sun)])
