"""CPU tests of the flux boundaries (prb_set_flux_boundaries): the FP64 restatement (tests/boundary_flux_oracle.py)
against the existing oracles with the default boundaries, against closed forms (isothermal, transparent, perfectly
reflecting columns), and the Python argument checks of Engine.set_flux_boundaries and Atmosphere.columnFluxes."""
import numpy as np
import pytest

from oracle import physics as ph
from pyrad_b200 import classes as C
from pyrad_b200 import engine as eng
from tests import band_flux_oracle as BO
from tests import boundary_flux_oracle as XO
from tests import flux_oracle as FO

RMIN, RMAX, RES = 0.0, 2500.0, 1.0          # includes the 0 cm-1 point, where Planck is 0/0 = NaN
NU = ph.x_axis(RMIN, RMAX, RES)
TABLE = ([0.0, 800.0, 1000.0, 1100.0, 1500.0], [1.0, 0.95, 0.0, 0.7, 1.0])   # reaches 0 and 1 inside the axis


def random_column(L, seed, n=NU.size):
    rng = np.random.default_rng(seed)
    k = 10.0 ** rng.uniform(-8, 0, (L, n))
    depth = rng.uniform(1e4, 1e5, L)
    T = rng.uniform(200, 300, L)
    return k, depth, T


def pi_int_planck(T):
    return ph.integrate_spectrum(ph.planck_wavenumber(NU, T), ph.pi, RES)


@pytest.mark.parametrize("n_mu", [1, 3, 4])
@pytest.mark.parametrize("eps", [None, 1.0, ([500.0], [1.0])])
@pytest.mark.parametrize("reflection", ["lambertian", "specular"])
def test_black_surface_and_cold_top_give_the_existing_oracles_bit_for_bit(n_mu, eps, reflection):
    k, depth, T = random_column(5, 11)
    rng = np.random.default_rng(n_mu)
    mu, w = rng.uniform(0.1, 1.0, n_mu), rng.uniform(0.05, 0.5, n_mu)
    got = XO.boundary_fluxes(k, depth, T, 288.0, NU, RES, mu, w, eps, reflection, 0.0)
    ref = FO.column_fluxes(k, depth, T, 288.0, NU, RES, mu, w)
    for a, b in zip(got, ref):
        assert a.tobytes() == b.tobytes()
    edges = [0.0, 10.0, 630.0, 700.0, 2000.0, 2400.5]
    got = XO.boundary_band_fluxes(k, depth, T, 288.0, NU, RES, mu, w, edges, eps, reflection, 0.0)
    ref = BO.band_fluxes(k, depth, T, 288.0, NU, RES, mu, w, edges)
    for a, b in zip(got, ref):
        assert a.tobytes() == b.tobytes()


@pytest.mark.parametrize("eps", [0.3, TABLE, ([1200.0], [0.0])])
@pytest.mark.parametrize("reflection", ["lambertian", "specular"])
@pytest.mark.parametrize("n_mu", [1, 3, 4])
def test_isothermal_column_with_an_isothermal_top_is_isotropic(eps, reflection, n_mu):
    """T_l = T_s = T_top: every radiance is B whatever the surface reflects, and with sum w mu = 1/2 every level flux
    in either direction is pi integral B."""
    k, depth, _ = random_column(6, 3)
    mu, w = FO.gauss_legendre_01(n_mu)
    up, down, ru, rd = XO.boundary_fluxes(k, depth, np.full(6, 250.0), 250.0, NU, RES, mu, w, eps, reflection, 250.0)
    ref = pi_int_planck(250.0)
    np.testing.assert_allclose(up, ref, rtol=1e-12)
    np.testing.assert_allclose(down, ref, rtol=1e-12)
    b = ph.planck_wavenumber(NU, 250.0)
    for rows in (ru, rd):
        np.testing.assert_allclose(rows[:, 1:], np.broadcast_to(b[1:], (n_mu, NU.size - 1)), rtol=1e-12)


@pytest.mark.parametrize("eps", [0.6, TABLE])
@pytest.mark.parametrize("t_top", [2.725, 250.0])
def test_transparent_column_shows_the_surface_and_the_reflected_top(eps, t_top):
    """k = 0, Lambertian, sum w mu = 1/2: the surface reflects 1 - eps of B(T_top), so I_up = eps B(T_s) + (1 - eps)
    B(T_top) at every point and node, and I_down = B(T_top)."""
    L = 4
    mu, w = FO.gauss_legendre_01(3)
    up, down, ru, rd = XO.boundary_fluxes(np.zeros((L, NU.size)), np.full(L, 1e5), np.linspace(290, 210, L), 288.0, NU,
                                          RES, mu, w, eps, "lambertian", t_top)
    e = XO.emissivity(NU, eps)
    with np.errstate(invalid="ignore", over="ignore"):
        bt = ph.planck_wavenumber(NU, t_top)
    expect = e * ph.planck_wavenumber(NU, 288.0) + (1 - e) * bt
    np.testing.assert_allclose(ru[:, 1:], np.broadcast_to(expect[1:], (3, NU.size - 1)), rtol=1e-12)
    np.testing.assert_allclose(rd[:, 1:], np.broadcast_to(bt[1:], (3, NU.size - 1)), rtol=1e-12)
    np.testing.assert_allclose(up, ph.integrate_spectrum(expect, ph.pi, RES), rtol=1e-12)
    np.testing.assert_allclose(down, ph.integrate_spectrum(bt, ph.pi, RES), rtol=1e-12)


@pytest.mark.parametrize("t_top", [0.0, 250.0])
def test_perfect_lambertian_reflector_sends_back_what_comes_down(t_top):
    k, depth, T = random_column(5, 7)
    mu, w = FO.gauss_legendre_01(3)
    up, down, _, _ = XO.boundary_fluxes(k, depth, T, 288.0, NU, RES, mu, w, 0.0, "lambertian", t_top)
    np.testing.assert_allclose(up[0], down[0], rtol=1e-12)
    assert up[0] > 0


def test_perfect_specular_reflector_over_a_transparent_column_returns_each_node_its_own_radiance():
    L = 3
    mu, w = FO.gauss_legendre_01(3)
    _, _, ru, rd = XO.boundary_fluxes(np.zeros((L, NU.size)), np.full(L, 1e5), np.full(L, 250.0), 288.0, NU, RES, mu,
                                      w, 0.0, "specular", 200.0)
    np.testing.assert_array_equal(ru[:, 1:], rd[:, 1:])


def test_grey_surface_lowers_the_outgoing_flux_and_the_surface_net_flux():
    k, depth, T = random_column(6, 5)
    mu, w = FO.gauss_legendre_01(3)
    black = FO.column_fluxes(k, depth, T, 288.0, NU, RES, mu, w)
    grey = XO.boundary_fluxes(k, depth, T, 288.0, NU, RES, mu, w, TABLE, "lambertian", 2.725)
    assert grey[0][-1] < black[0][-1]
    assert grey[0][0] - grey[1][0] < black[0][0] - black[1][0]


def test_emissivity_is_np_interp_rounded_to_fp32():
    e = XO.emissivity(NU, TABLE)
    np.testing.assert_array_equal(e, np.interp(NU, *TABLE).astype(np.float32))
    assert e[0] == 1.0 and e.min() < 0.01 and e[-1] == 1.0
    np.testing.assert_array_equal(XO.emissivity(NU, ([300.0], [0.25])), np.full(NU.size, 0.25))
    np.testing.assert_array_equal(XO.emissivity(NU, None), np.ones(NU.size))


def test_flux_boundary_args():
    nu, eps, refl, t = eng.flux_boundary_args()
    assert nu.size == eps.size == 0 and refl == 0 and t == 0.0
    nu, eps, refl, t = eng.flux_boundary_args(0.9, "specular", 2.725)
    assert list(nu) == [0.0] and list(eps) == [0.9] and refl == 1 and t == 2.725
    nu, eps, _, _ = eng.flux_boundary_args(TABLE)
    assert list(nu) == TABLE[0] and list(eps) == TABLE[1]


@pytest.mark.parametrize("kw", [
    dict(emissivity=1.5), dict(emissivity=-0.1), dict(emissivity=np.nan),
    dict(emissivity=([0.0, 1.0], [0.5])), dict(emissivity=([1.0, 0.0], [0.5, 0.5])),
    dict(emissivity=([0.0, 0.0], [0.5, 0.5])), dict(emissivity=([0.0, np.inf], [0.5, 0.5])),
    dict(emissivity=([0.0, 1.0], [0.5, np.nan])), dict(emissivity=([], [])), dict(emissivity=([[0.0]], [[0.5]])),
    dict(emissivity=(1.0, 2.0, 3.0)), dict(reflection="mirror"), dict(reflection=1),
    dict(t_top=-1.0), dict(t_top=np.inf), dict(t_top=np.nan)])
def test_flux_boundary_args_reject_bad_input(kw):
    with pytest.raises(ValueError):
        eng.flux_boundary_args(**kw)


@pytest.mark.parametrize("kw", [dict(surfaceEmissivity=2.0), dict(reflection="glossy"), dict(topTemperature=-3.0)])
def test_column_fluxes_rejects_bad_boundaries_before_the_column_runs(kw):
    atm = C.Atmosphere("empty")              # no layers: the column itself would fail, with another message
    with pytest.raises(ValueError, match="emissivity|reflection|t_top"):
        atm.columnFluxes(288.0, **kw)
