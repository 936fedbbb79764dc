"""TEST INFRASTRUCTURE ONLY -- FP64 numpy restatement of the band fluxes (prb_atmosphere_band_fluxes).

The column fluxes of tests/flux_oracle.py (the reference's Layer.transmission along a slant path and its
integrateSpectrum), with the level sums split by wavenumber band.  Same fold, same non-finite rule.
"""
import numpy as np

from oracle import physics as ph
from tests.flux_oracle import FLT_MAX


def band_fluxes(k, depth_cm, T, t_surface, nu, res, mu, weights, edges):
    """The fluxes of column_fluxes split by wavenumber band: grid point nu belongs to band b when
    edges[b] <= nu < edges[b+1] (np.searchsorted(edges, nu, side="right") - 1); points outside [edges[0], edges[-1])
    count nowhere.  The same FP64 fold and non-finite rule as column_fluxes.

    Returns (band_up, band_down), (n_bands, L+1) each."""
    L = len(depth_cm)
    nu = np.asarray(nu, dtype=np.float64)
    edges = np.asarray(edges, dtype=np.float64)
    nb = edges.size - 1
    mu, weights = np.atleast_1d(np.asarray(mu, dtype=np.float64)), np.atleast_1d(np.asarray(weights, dtype=np.float64))
    idx = np.searchsorted(edges, nu, side="right") - 1
    sel = (idx >= 0) & (idx < nb)
    planck = [ph.planck_wavenumber(nu, T[l]) for l in range(L)]
    up, down = np.zeros((nb, L + 1)), np.zeros((nb, L + 1))

    def add(flux, j, w, m, I):
        I = np.where(np.abs(I) <= FLT_MAX, I, 0.0)
        flux[:, j] += 2 * ph.pi * w * m * np.bincount(idx[sel], weights=I[sel], minlength=nb) * res

    for m, w in zip(mu, weights):
        I = ph.planck_wavenumber(nu, t_surface)
        add(up, 0, w, m, I)
        for l in range(L):
            t = np.exp(-np.asarray(k[l], dtype=np.float64) * depth_cm[l] / m)
            I = ph.transmission(t, I, planck[l])
            add(up, l + 1, w, m, I)
        I = np.zeros_like(nu)
        for l in range(L - 1, -1, -1):
            t = np.exp(-np.asarray(k[l], dtype=np.float64) * depth_cm[l] / m)
            I = ph.transmission(t, I, planck[l])
            add(down, l, w, m, I)
    return up, down
