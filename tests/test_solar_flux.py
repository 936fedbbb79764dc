"""CPU tests of the solar beam (prb_set_solar_source): the FP64 restatement (tests/solar_flux_oracle.py) against the
boundary oracle without sunlight, against closed forms (transparent columns, one absorbing layer over a black surface),
the zero outside the irradiance table, and the Python argument checks of Engine.set_solar_source and
Atmosphere.columnFluxes."""
import numpy as np
import pytest

from oracle import physics as ph
from pyrad_b200 import classes as C
from pyrad_b200 import engine as eng
from tests import boundary_flux_oracle as XO
from tests import flux_oracle as FO
from tests import solar_flux_oracle as SO

RMIN, RMAX, RES = 0.0, 2500.0, 1.0          # includes the 0 cm-1 point, where Planck is 0/0 = NaN
NU = ph.x_axis(RMIN, RMAX, RES)
EPS_TABLE = ([0.0, 800.0, 1000.0, 1100.0, 1500.0], [1.0, 0.95, 0.0, 0.7, 1.0])   # reaches 0 and 1 inside the axis
SUN = ([0.0, 700.0, 1500.0, 2600.0], [0.0, 2e-3, 1.5e-2, 4e-2])                   # W m-2 (cm-1)-1, covers the axis


def random_column(L, seed, n=NU.size):
    rng = np.random.default_rng(seed)
    k = 10.0 ** rng.uniform(-8, 0, (L, n))
    depth = rng.uniform(1e4, 1e5, L)
    T = rng.uniform(200, 300, L)
    return k, depth, T


def transparent(L=4):
    return np.zeros((L, NU.size)), np.full(L, 1e5), np.linspace(290, 210, L)


@pytest.mark.parametrize("n_mu", [1, 3, 4])
@pytest.mark.parametrize("eps", [None, 0.4, EPS_TABLE])
@pytest.mark.parametrize("reflection", ["lambertian", "specular"])
@pytest.mark.parametrize("t_top", [0.0, 250.0])
def test_a_dark_sun_gives_the_boundary_oracle_bit_for_bit(n_mu, eps, reflection, t_top):
    k, depth, T = random_column(5, 11)
    rng = np.random.default_rng(n_mu)
    mu, w = rng.uniform(0.1, 1.0, n_mu), rng.uniform(0.05, 0.5, n_mu)
    dark = ([0.0, 3000.0], [0.0, 0.0])
    got = SO.solar_fluxes(k, depth, T, 288.0, NU, RES, mu, w, dark, 0.3, eps, reflection, t_top)
    ref = XO.boundary_fluxes(k, depth, T, 288.0, NU, RES, mu, w, eps, reflection, t_top)
    for a, b in zip(got, ref):
        assert a.tobytes() == b.tobytes()
    edges = [0.0, 10.0, 630.0, 700.0, 2000.0, 2400.5]
    got = SO.solar_band_fluxes(k, depth, T, 288.0, NU, RES, mu, w, edges, dark, 0.3, eps, reflection, t_top)
    ref = XO.boundary_band_fluxes(k, depth, T, 288.0, NU, RES, mu, w, edges, eps, reflection, t_top)
    for a, b in zip(got, ref):
        assert a.tobytes() == b.tobytes()


@pytest.mark.parametrize("mu_sun", [1.0, 0.5, 0.05])
@pytest.mark.parametrize("eps", [None, 0.3, EPS_TABLE])
@pytest.mark.parametrize("reflection", ["lambertian", "specular"])
def test_transparent_column_adds_the_beam_and_its_reflection(mu_sun, eps, reflection):
    """k = 0: flux_down gains mu_sun sum S res at every level, and flux_up mu_sun sum (1 - eps) S res (Lambertian with
    Gauss-Legendre nodes, sum w mu = 1/2; specular for any quadrature); the solar part of the net flux at the surface
    is -mu_sun sum eps S res."""
    k, depth, T = transparent()
    mu, w = FO.gauss_legendre_01(3) if reflection == "lambertian" else (np.array([0.2, 0.9]), np.array([0.7, 0.3]))
    s = SO.irradiance(NU, SUN)
    e = XO.emissivity(NU, eps)
    dark = SO.solar_fluxes(k, depth, T, 288.0, NU, RES, mu, w, None, mu_sun, eps, reflection)
    lit = SO.solar_fluxes(k, depth, T, 288.0, NU, RES, mu, w, SUN, mu_sun, eps, reflection)
    np.testing.assert_allclose(lit[1] - dark[1], mu_sun * np.sum(s) * RES, rtol=1e-9)
    np.testing.assert_allclose(lit[0] - dark[0], mu_sun * np.sum((1 - e) * s) * RES, rtol=1e-9, atol=1e-12)
    net = (lit[1][0] - lit[0][0]) - (dark[1][0] - dark[0][0])
    np.testing.assert_allclose(net, mu_sun * np.sum(e * s) * RES, rtol=1e-9)
    np.testing.assert_array_equal(lit[3], dark[3])                     # the beam is not a node


def test_one_absorbing_layer_over_a_black_surface():
    """The beam's surface flux is mu_sun sum S exp(-tau / mu_sun) res, tau = k depth."""
    L, mu_sun = 1, 0.5
    k = np.full((L, NU.size), 2e-5)
    depth = np.array([1e4])                                              # tau = 0.2
    mu, w = FO.gauss_legendre_01(3)
    dark = SO.solar_fluxes(k, depth, [250.0], 288.0, NU, RES, mu, w)
    lit = SO.solar_fluxes(k, depth, [250.0], 288.0, NU, RES, mu, w, SUN, mu_sun)
    s = SO.irradiance(NU, SUN)
    np.testing.assert_allclose(lit[1][0] - dark[1][0], mu_sun * np.sum(s * np.exp(-0.2 / mu_sun)) * RES, rtol=1e-12)
    np.testing.assert_allclose(lit[1][1] - dark[1][1], mu_sun * np.sum(s) * RES, rtol=1e-12)
    for a, b in ((lit[0], dark[0]), (lit[2], dark[2]), (lit[3], dark[3])):   # a black surface reflects nothing
        assert a.tobytes() == b.tobytes()
    np.testing.assert_allclose(SO.beam_flux_down(k, depth, NU, RES, SUN, mu_sun), lit[1] - dark[1], rtol=1e-12)


def test_a_table_over_part_of_the_axis_is_zero_outside_it():
    part = ([600.0, 900.0, 1200.0], [1e-2, 3e-2, 2e-2])
    s = SO.irradiance(NU, part)
    inside = (NU >= 600.0) & (NU <= 1200.0)
    assert np.all(s[~inside] == 0) and np.all(s[inside] > 0)
    np.testing.assert_array_equal(s[inside], np.interp(NU[inside], *part).astype(np.float32))
    np.testing.assert_array_equal(SO.irradiance([600.0, 1200.0], part), np.float32([1e-2, 2e-2]))
    np.testing.assert_array_equal(SO.irradiance(NU, None), np.zeros(NU.size))
    k, depth, T = transparent(2)
    mu, w = FO.gauss_legendre_01(2)
    lit = SO.solar_band_fluxes(k, depth, T, 288.0, NU, RES, mu, w, [0.0, 600.0, 1201.0, 2501.0], part, 1.0)
    dark = SO.solar_band_fluxes(k, depth, T, 288.0, NU, RES, mu, w, [0.0, 600.0, 1201.0, 2501.0])
    d = lit[1] - dark[1]
    assert np.all(d[0] == 0) and np.all(d[2] == 0)
    np.testing.assert_allclose(d[1], np.sum(s) * RES, rtol=1e-12)


def test_solar_source_args():
    nu, s, m = eng.solar_source_args()
    assert nu.size == s.size == 0 and m == 1.0
    nu, s, m = eng.solar_source_args(SUN, 0.5)
    assert list(nu) == SUN[0] and list(s) == SUN[1] and m == 0.5
    nu, s, m = eng.solar_source_args(np.array([[1.0, 2.0], [0.0, 0.0]]), 1)
    assert list(nu) == [1.0, 2.0] and list(s) == [0.0, 0.0] and m == 1.0


@pytest.mark.parametrize("kw", [
    dict(irradiance=([0.0, np.nan], [1.0, 1.0])), dict(irradiance=([0.0, np.inf], [1.0, 1.0])),
    dict(irradiance=([1.0, 0.0], [1.0, 1.0])), dict(irradiance=([1.0, 1.0], [1.0, 1.0])),
    dict(irradiance=([0.0, 1.0], [1.0, -1e-3])), dict(irradiance=([0.0, 1.0], [1.0, np.nan])),
    dict(irradiance=([0.0, 1.0], [1.0, np.inf])), dict(irradiance=([0.0], [1.0])),
    dict(irradiance=([0.0, 1.0, 2.0], [1.0, 1.0])), dict(irradiance=([[0.0, 1.0]], [[1.0, 1.0]])),
    dict(irradiance=1.0), dict(irradiance=([0.0, 1.0], [1.0, 1.0], [2.0, 2.0])),
    dict(irradiance=SUN, mu_sun=0.0), dict(irradiance=SUN, mu_sun=-0.5), dict(irradiance=SUN, mu_sun=1.01),
    dict(irradiance=SUN, mu_sun=np.nan), dict(irradiance=SUN, mu_sun=np.inf)])
def test_solar_source_args_reject_bad_input(kw):
    with pytest.raises(ValueError):
        eng.solar_source_args(**kw)


@pytest.mark.parametrize("kw", [dict(solarIrradiance=([0.0, 1.0], [1.0, -1.0])), dict(solarIrradiance=([0.0], [1.0])),
                                dict(solarIrradiance=SUN, solarMu=0.0), dict(solarIrradiance=SUN, solarMu=2.0)])
def test_column_fluxes_rejects_a_bad_sun_before_the_column_runs(kw):
    atm = C.Atmosphere("empty")              # no layers: the column itself would fail, with another message
    with pytest.raises(ValueError, match="irradiance|mu_sun"):
        atm.columnFluxes(288.0, **kw)
