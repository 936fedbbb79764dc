"""CPU tests of the layer kernels' FP64 restatement (tests/kernel_oracle.py): the O(L) formula against brute force, the
closed forms of a transparent column, identical columns and one opaque layer, and the argument validation of
Engine.atmosphere_layer_kernels and Atmosphere.columnKernels that runs before any device call."""
import numpy as np
import pytest

from oracle import physics as ph
from pyrad_b200 import classes as C
from pyrad_b200 import engine as eng
from tests import flux_oracle as FO
from tests import kernel_oracle as KO


def random_pair(rng, L, n=400, nu0=500.0, step=0.5):
    nu = nu0 + step * np.arange(n)
    base = {"k": rng.uniform(0, 2, (L, n)) * 10.0 ** rng.uniform(-4, 1, (L, 1)), "depth_cm": rng.uniform(0.5, 2, L),
            "T": rng.uniform(200, 300, L), "t_surface": 290.0}
    kind = rng.integers(3)
    cur = {"k": base["k"] * (1 + (kind == 1) * rng.uniform(-0.1, 0.1, (L, 1))), "depth_cm": base["depth_cm"] * (
        1 + (kind == 2) * 0.1), "T": base["T"] + (kind == 0) * 1.0 + rng.uniform(-0.5, 0.5, L), "t_surface": 291.0}
    return nu, base, cur


@pytest.mark.parametrize("seed", range(12))
def test_the_o_l_formula_equals_brute_force(seed):
    rng = np.random.default_rng(seed)
    L = 1 + seed % 8
    nu, base, cur = random_pair(rng, L)
    mu, wt = FO.gauss_legendre_01(1 + seed % 4)
    edges = np.sort(rng.uniform(nu[0] - 5, nu[-1] + 5, 1 + seed % 5))
    edges = np.concatenate([[nu[0] - 1], edges, [nu[-1] + 1]])
    t_top = 2.725 if seed % 3 == 0 else 0.0
    got = KO.layer_kernels(base, cur, nu, 0.5, mu, wt, edges, t_top)
    ref = KO.brute_force(base, cur, nu, 0.5, mu, wt, edges, t_top)
    scale = np.abs(KO.boundary_fluxes(base["k"], base["depth_cm"], base["T"], base["t_surface"], nu, 0.5, mu, wt, edges,
                                      t_top)).sum()
    for g, r, a in ((got[0], ref[0], got[2]), (got[1], ref[1], got[3])):
        np.testing.assert_array_less(np.abs(g - r), 1e-10 * (np.abs(r) + a) + 1e-14 * scale + 1e-300)


def test_a_transparent_column_gives_only_the_surface_entry():
    nu = np.linspace(100.0, 2000.0, 3000)
    L = 5
    base = {"k": np.zeros((L, nu.size)), "depth_cm": np.ones(L), "T": np.full(L, 250.0), "t_surface": 288.0}
    cur = dict(base, T=base["T"] + 1, t_surface=289.0)
    mu, wt = FO.gauss_legendre_01(3)                               # sum w mu = 1/2
    res = nu[1] - nu[0]
    up, down, _, _ = KO.layer_kernels(base, cur, nu, res, mu, wt, [nu[0], nu[-1] + 1])
    assert np.all(up[:, 1:] == 0) and np.all(down == 0)
    d_b = ph.planck_wavenumber(nu, 289.0) - ph.planck_wavenumber(nu, 288.0)
    np.testing.assert_allclose(up[0, 0], ph.pi * d_b.sum() * res, rtol=1e-12)


def test_identical_columns_give_zero():
    nu, base, _ = random_pair(np.random.default_rng(7), 6)
    mu, wt = FO.gauss_legendre_01(2)
    for x in KO.layer_kernels(base, base, nu, 0.5, mu, wt, [nu[0], 600.0, nu[-1] + 1])[:2]:
        assert np.all(x == 0)


def test_a_single_opaque_layer():
    """One black layer: the top sees B(T_1) only, so its 1 K kernel is pi (B(T+1) - B(T)) integrated, and the
    surface's entry is 0; downward likewise."""
    nu = np.linspace(500.0, 1500.0, 2001)
    res = nu[1] - nu[0]
    base = {"k": np.full((1, nu.size), 1e4), "depth_cm": np.ones(1), "T": np.array([260.0]), "t_surface": 288.0}
    cur = dict(base, T=np.array([261.0]), t_surface=290.0)
    mu, wt = FO.gauss_legendre_01(3)
    up, down, _, _ = KO.layer_kernels(base, cur, nu, res, mu, wt, [nu[0], nu[-1] + 1])
    exp = ph.pi * (ph.planck_wavenumber(nu, 261.0) - ph.planck_wavenumber(nu, 260.0)).sum() * res
    np.testing.assert_allclose(up[0], [0.0, exp], rtol=1e-12, atol=0)
    np.testing.assert_allclose(down[0], [0.0, exp], rtol=1e-12, atol=0)


@pytest.mark.parametrize("mu, wt, edges", [
    ([0.5, 0.5], [1.0], [1.0, 2.0]),
    ([0.1, 0.2, 0.3, 0.4, 0.5], [1.0] * 5, [1.0, 2.0]),
    ([0.0], [1.0], [1.0, 2.0]),
    ([0.5], [-1.0], [1.0, 2.0]),
    ([0.5], [1.0], [2.0, 1.0]),
    ([0.5], [1.0], [1.0]),
    ([0.5], [1.0], [1.0, np.nan]),
    ([0.5], [1.0], [[1.0, 2.0]]),
])
def test_engine_wrapper_rejects_bad_arguments_before_the_library(mu, wt, edges):
    e = eng.Engine.__new__(eng.Engine)                             # no device: the checks come first
    with pytest.raises(ValueError, match="atmosphere_layer_kernels"):
        e.atmosphere_layer_kernels(mu, wt, edges)


def test_an_opaque_layer_keeps_every_node():
    """T' - T where the layer is opaque along a slant node: T underflows and expm1(-dtau / mu) overflows, so the product
    form alone is 0 * inf = NaN and would drop the node; the difference must stay finite (here 0) and the kernel must
    be the opaque layer's pi (B' - B) res for any quadrature with sum w mu = 1/2."""
    dt = KO.transmittance_difference(np.array([1e4, 1.0]), np.array([-100.0, 1e-3]), 0.1)
    assert np.all(np.isfinite(dt)) and dt[0] == 0
    np.testing.assert_allclose(dt[1], np.exp(-10.0) * np.expm1(-1e-2), rtol=1e-14)
    nu = np.linspace(1.0, 40.0, 500)
    res = nu[1] - nu[0]
    base = {"k": np.full((1, nu.size), 1e-2), "depth_cm": np.array([1e6]), "T": np.array([280.0]), "t_surface": 288.0}
    cur = dict(base, k=base["k"] * 0.99, T=np.array([281.0]))
    exp = ph.pi * (ph.planck_wavenumber(nu, 281.0) - ph.planck_wavenumber(nu, 280.0)).sum() * res
    for n in (1, 3):
        mu, wt = FO.gauss_legendre_01(n)
        down = KO.layer_kernels(base, cur, nu, res, mu, wt, [0.0, 41.0])[1]
        np.testing.assert_allclose(down[0, 1], exp, rtol=1e-12)


def _layers(name, n, rmax=640.0, T=280.0):
    atm = C.Atmosphere(name)
    for i in range(n):
        atm.addLayer(1e5, T - 10 * i, 800.0 / (i + 1), 600.0, rmax, dynamicResolution=False)
    return atm


def test_column_kernels_rejects_bad_arguments_before_the_columns_run(monkeypatch):
    monkeypatch.setattr(C.Layer, "hasAtmosphere", False)          # Layer keeps the first atmosphere class-wide
    atm = C.Atmosphere("empty")
    with pytest.raises(ValueError, match="Atmosphere"):
        atm.columnKernels(288.0, "not a column")
    with pytest.raises(ValueError, match="layers"):
        atm.columnKernels(288.0, C.Atmosphere("other"))
    with pytest.raises(ValueError):
        atm.columnKernels(288.0, C.Atmosphere("other"), topTemperature=-1.0)
    two = _layers("two", 2)
    with pytest.raises(ValueError, match="as many layers"):
        two.columnKernels(288.0, _layers("three", 3))
    with pytest.raises(ValueError, match="same grid"):
        two.columnKernels(288.0, _layers("wider", 2, rmax=650.0))
    with pytest.raises(ValueError, match="bands"):
        two.columnKernels(288.0, _layers("warm", 2, T=281.0), bands=[640.0, 600.0])
    with pytest.raises(ValueError, match="quadrature"):
        two.columnKernels(288.0, _layers("warm", 2, T=281.0), mu=[0.5, 0.6], weights=[1.0])
