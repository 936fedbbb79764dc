"""TEST INFRASTRUCTURE ONLY -- FP64 numpy restatement of the column fluxes (prb_atmosphere_fluxes).

The reference ships no fluxes, no downward pass and no slant paths (SURVEY.md section 3.5).  What is restated here is
the reference's own layer step, Layer.transmission (pyradClasses.py:784-787, ``oracle.physics.transmission``), applied
along a slant path (optical depth k * depth / mu), and its integral, integrateSpectrum (pyradClasses.py:26-29:
sum(nan_to_num(I)) * res).  Built from the oracle's functions so that mu = 1 reproduces the oracle's layer-by-layer
transmission chain bit for bit.
"""
import numpy as np

from oracle import physics as ph

FLT_MAX = float(np.finfo(np.float32).max)


def column_fluxes(k, depth_cm, T, t_surface, nu, res, mu, weights):
    """Hemispheric fluxes and slant radiances of a column, layers 0..L-1 from the bottom up over a blackbody surface.

    k: (L, n) absorption coefficients (or a list of L rows); depth_cm, T: per layer; nu: the wavenumber axis (Planck's
    argument, the layers' linspace or a chunk of it); res: the integration step; mu, weights: the angular quadrature.
    Per node mu_i: upward from B(nu, t_surface) at level 0, downward from 0 at level L, through layer l with
    I <- T I + (1 - T) B(nu, T_l), T = exp(-k_l depth_l / mu_i).  Level j is the boundary below layer j (0 = surface,
    L = top).  F[j] = 2 pi sum_i w_i mu_i sum_nu nan_to_num(I_i(nu, level j)) res -- with sum_i w_i mu_i = 1/2 (Gauss-
    Legendre on [0, 1]) an isotropic field gives pi B.

    NaN counts as 0 (integrateSpectrum's nan_to_num), and so does a value beyond the FP32 range: only the reference's
    negative Doppler widths next to 0 cm-1 make k < 0 and exp(-k u) overflow, where nan_to_num would add +-1.8e308;
    the device's FP32 fold has +-inf there and counts it as 0.

    Returns (flux_up, flux_down, rad_up_top, rad_down_surface): (L+1,) each, then (n_mu, n) each."""
    L = len(depth_cm)
    nu = np.asarray(nu, dtype=np.float64)
    mu, weights = np.atleast_1d(np.asarray(mu, dtype=np.float64)), np.atleast_1d(np.asarray(weights, dtype=np.float64))
    planck = [ph.planck_wavenumber(nu, T[l]) for l in range(L)]
    up, down = np.zeros(L + 1), np.zeros(L + 1)
    rad_up, rad_down = [], []

    def add(flux, j, w, m, I):
        flux[j] += 2 * ph.pi * w * m * np.sum(np.where(np.abs(I) <= FLT_MAX, I, 0.0)) * res

    for m, w in zip(mu, weights):
        I = ph.planck_wavenumber(nu, t_surface)
        add(up, 0, w, m, I)
        for l in range(L):
            t = np.exp(-np.asarray(k[l], dtype=np.float64) * depth_cm[l] / m)
            I = ph.transmission(t, I, planck[l])
            add(up, l + 1, w, m, I)
        rad_up.append(I)
        I = np.zeros_like(nu)
        for l in range(L - 1, -1, -1):
            t = np.exp(-np.asarray(k[l], dtype=np.float64) * depth_cm[l] / m)
            I = ph.transmission(t, I, planck[l])
            add(down, l, w, m, I)
        rad_down.append(I)
    return up, down, np.array(rad_up), np.array(rad_down)


def gauss_legendre_01(n):
    """n-node Gauss-Legendre rule on [0, 1]: (mu, weights), sum of the weights 1."""
    x, w = np.polynomial.legendre.leggauss(n)
    return (x + 1) / 2, w / 2
