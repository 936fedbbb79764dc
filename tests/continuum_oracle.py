"""TEST INFRASTRUCTURE ONLY -- FP64 numpy restatement of the water-vapour continuum (prb_set_continuum).

PyRad has no continuum.  The engine takes one in MT_CKD's form (self and foreign coefficients and the self coefficient's
temperature exponent, at a reference temperature and pressure) and adds, for layer l and every point nu of the Planck axis,

    k_c,l(nu) = n_l rho_l R(nu, T_l) [x_l (t_ref/T_l)^n(nu) C_s(nu) + (1 - x_l) C_f(nu)]

to row l of the column's k matrix before the fold, with n_l = x_l P_l / 1e4 / kB / T_l (absCoef's number density factor,
pyradClasses.py:581-583), rho_l = (P_l / p_ref)(t_ref / T_l) and R(nu, T) = nu tanh(c2 nu / 2T).  Column results are the
existing flux oracles (tests/flux_oracle.py, tests/band_flux_oracle.py) on k + k_c.
"""
import numpy as np

from oracle import physics as ph

C2 = 100 * ph.h * ph.c / ph.k           # cm K, the engine's c2


def number_density(x, P, T):
    """Molecules cm-3 of a gas at mole fraction x (P in hPa, T in K), left to right as absCoef."""
    return x * P / 1E4 / ph.k / T


def radiation_term(nu, T):
    """R(nu, T) = nu tanh(c2 nu / 2T) in cm-1; R(0) = 0."""
    nu = np.asarray(nu, dtype=np.float64)
    return nu * np.tanh(C2 * nu / (2 * T))


def coefficients(nu, table):
    """(C_s, C_f, n) on the axis nu: np.interp of the table, 0 outside it for the two coefficients, clamped for n."""
    tn = np.asarray(table["nu"], dtype=np.float64)
    cs = np.interp(nu, tn, np.asarray(table["self"], dtype=np.float64), left=0.0, right=0.0)
    cf = np.interp(nu, tn, np.asarray(table["foreign"], dtype=np.float64), left=0.0, right=0.0)
    n = np.interp(nu, tn, np.asarray(table["texp"], dtype=np.float64))
    return cs, cf, n


def layer_continuum(nu, T, P, x, table):
    """k_c of one layer on the axis nu, in cm-1."""
    t_ref, p_ref = float(table.get("t_ref", 296.0)), float(table.get("p_ref", 1013.0))
    cs, cf, n = coefficients(nu, table)
    rho = (P / p_ref) * (t_ref / T)
    return number_density(x, P, T) * rho * radiation_term(nu, T) * (x * (t_ref / T) ** n * cs + (1 - x) * cf)


def continuum(nu, T, P, x, table):
    """(L, n) k_c of every layer of a column: T, P, x per layer."""
    return np.array([layer_continuum(nu, T[l], P[l], x[l], table) for l in range(len(T))])


def synthetic_table(seed, lo, hi, spacing=10.0):
    """A table in MT_CKD's form over [lo, hi] with about `spacing` cm-1 between entries: coefficients log-uniform in
    [1e-27, 1e-21] cm2 molecule-1 (cm-1)-1, exponents uniform in [0, 6].  A synthetic table, not MT_CKD's."""
    rng = np.random.default_rng(seed)
    m = max(2, int(round((hi - lo) / spacing)) + 1)
    nu = np.linspace(lo, hi, m)
    return {"nu": nu, "self": 10.0 ** rng.uniform(-27, -21, m), "foreign": 10.0 ** rng.uniform(-27, -21, m),
            "texp": rng.uniform(0.0, 6.0, m)}


def synthetic_mole_fractions(seed, L):
    """L mole fractions, log-uniform from 1e-6 to 0.03."""
    return 10.0 ** np.random.default_rng(seed).uniform(-6, np.log10(0.03), L)
