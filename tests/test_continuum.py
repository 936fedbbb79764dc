"""CPU tests of the water-vapour continuum's FP64 restatement (tests/continuum_oracle.py) and of the argument checks of
engine.continuum_args."""
import numpy as np
import pytest

from pyrad_b200 import engine as eng
from tests import continuum_oracle as CO

TABLE = {"nu": [500.0, 800.0, 1000.0, 1400.0], "self": [2e-22, 5e-23, 1e-23, 3e-23],
         "foreign": [1e-24, 4e-25, 2e-25, 6e-25], "texp": [4.0, 5.5, 6.0, 3.0]}


def test_radiation_term_limits():
    T = 250.0
    nu = np.array([1e-6, 1e-4, 1e-2, 0.1])
    np.testing.assert_allclose(CO.radiation_term(nu, T), CO.C2 * nu ** 2 / (2 * T), rtol=1e-6)
    assert CO.radiation_term(0.0, T) == 0.0
    big = np.array([3000.0, 5000.0])                  # c2 nu / 2T >= 8.6: tanh is 1 within 1e-7
    np.testing.assert_allclose(CO.radiation_term(big, T), big, rtol=1e-7)


def test_reference_state_reduces_to_number_density_times_r():
    nu = np.linspace(450.0, 1500.0, 2001)
    cs, cf, _ = CO.coefficients(nu, TABLE)
    for x in (1e-6, 0.01, 0.03):
        got = CO.layer_continuum(nu, 296.0, 1013.0, x, TABLE)
        ref = CO.number_density(x, 1013.0, 296.0) * CO.radiation_term(nu, 296.0) * (x * cs + (1 - x) * cf)
        np.testing.assert_allclose(got, ref, rtol=1e-14, atol=0)


def test_temperature_and_pressure_factors():
    nu = np.array([900.0])
    table = dict(TABLE, self=[0.0] * 4)                  # foreign only: rho scales it
    a = CO.layer_continuum(nu, 296.0, 500.0, 0.01, table)
    b = CO.layer_continuum(nu, 296.0, 1013.0, 0.01, table)
    np.testing.assert_allclose(a / b, (500.0 / 1013.0) ** 2, rtol=1e-12)       # n and rho both go with P
    table = dict(TABLE, foreign=[0.0] * 4, texp=[2.0] * 4)
    t = 250.0
    got = CO.layer_continuum(nu, t, 1013.0, 0.01, table)
    cs, _, _ = CO.coefficients(nu, table)
    ref = CO.number_density(0.01, 1013.0, t) * (296.0 / t) * CO.radiation_term(nu, t) * 0.01 * (296.0 / t) ** 2 * cs
    np.testing.assert_allclose(got, ref, rtol=1e-13)


def test_zero_mole_fraction_and_outside_the_table_give_zero():
    nu = np.concatenate([np.linspace(0.0, 499.99, 50), np.linspace(1400.01, 3000.0, 50)])
    assert np.all(CO.layer_continuum(nu, 260.0, 700.0, 0.02, TABLE) == 0.0)
    inside = np.linspace(500.0, 1400.0, 91)
    assert np.all(CO.layer_continuum(inside, 260.0, 700.0, 0.0, TABLE) == 0.0)
    assert np.all(CO.layer_continuum(inside, 260.0, 700.0, 0.02, TABLE) > 0.0)
    _, _, n = CO.coefficients(np.array([100.0, 2000.0]), TABLE)   # the exponent is clamped, not zeroed
    np.testing.assert_array_equal(n, [4.0, 3.0])


def test_linear_in_the_coefficients():
    nu = np.linspace(480.0, 1420.0, 777)
    T, P, x = 230.0, 400.0, 0.004
    only_self = dict(TABLE, foreign=[0.0] * 4)
    only_foreign = dict(TABLE, self=[0.0] * 4)
    both = CO.layer_continuum(nu, T, P, x, TABLE)
    np.testing.assert_allclose(CO.layer_continuum(nu, T, P, x, only_self) + CO.layer_continuum(nu, T, P, x, only_foreign),
                               both, rtol=1e-14)
    scaled = dict(TABLE, self=[3 * v for v in TABLE["self"]], foreign=[3 * v for v in TABLE["foreign"]])
    np.testing.assert_allclose(CO.layer_continuum(nu, T, P, x, scaled), 3 * both, rtol=1e-14)


def test_column_stacks_the_layers():
    nu = np.linspace(500.0, 1400.0, 11)
    T, P, x = [290.0, 250.0, 210.0], [900.0, 400.0, 50.0], [0.02, 0.0, 1e-6]
    k = CO.continuum(nu, T, P, x, TABLE)
    assert k.shape == (3, 11) and np.all(k[1] == 0)
    np.testing.assert_array_equal(k[2], CO.layer_continuum(nu, T[2], P[2], x[2], TABLE))


def test_synthetic_table_ranges():
    t = CO.synthetic_table(3, 590.0, 650.0)
    assert t["nu"].size == 7 and np.all(np.diff(t["nu"]) > 0)
    for key in ("self", "foreign"):
        assert np.all((t[key] >= 1e-27) & (t[key] <= 1e-21))
    assert np.all((t["texp"] >= 0) & (t["texp"] <= 6))
    x = CO.synthetic_mole_fractions(3, 50)
    assert np.all((x >= 1e-6) & (x <= 0.03))


def test_continuum_args_accepts_and_defaults():
    nu, cs, cf, tx, t_ref, p_ref, x = eng.continuum_args(TABLE, [0.01, 0.0, 1.0])
    np.testing.assert_array_equal(nu, TABLE["nu"])
    np.testing.assert_array_equal(cs, TABLE["self"])
    np.testing.assert_array_equal(cf, TABLE["foreign"])
    np.testing.assert_array_equal(tx, TABLE["texp"])
    assert (t_ref, p_ref) == (296.0, 1013.0)
    np.testing.assert_array_equal(x, [0.01, 0.0, 1.0])
    assert eng.continuum_args(dict(TABLE, t_ref=260.0, p_ref=500.0), [0.5])[4:6] == (260.0, 500.0)
    empty = eng.continuum_args()
    assert all(a.size == 0 for a in empty[:4]) and empty[6].size == 0
    assert eng.continuum_args(None, [0.5])[6].size == 0            # no table: the fractions are ignored


@pytest.mark.parametrize("table,x", [
    ([1.0, 2.0], [0.1]),                                           # not a dict
    ({k: v for k, v in TABLE.items() if k != "texp"}, [0.1]),      # a key missing
    (dict(TABLE, extra=[1.0]), [0.1]),                             # an unknown key
    (dict(TABLE, nu=[500.0]), [0.1]),                              # lengths differ
    ({"nu": [500.0], "self": [1e-22], "foreign": [1e-24], "texp": [4.0]}, [0.1]),   # one entry
    (dict(TABLE, nu=[500.0, 800.0, 800.0, 1400.0]), [0.1]),        # not strictly ascending
    (dict(TABLE, nu=[500.0, 800.0, np.nan, 1400.0]), [0.1]),
    (dict(TABLE, nu=[-np.inf, 800.0, 1000.0, 1400.0]), [0.1]),
    (dict(TABLE, self=[1e-22, -1e-30, 0.0, 0.0]), [0.1]),          # negative coefficient
    (dict(TABLE, foreign=[1e-22, np.nan, 0.0, 0.0]), [0.1]),
    (dict(TABLE, self=[1e-22, np.inf, 0.0, 0.0]), [0.1]),
    (dict(TABLE, texp=[1.0, np.inf, 0.0, 0.0]), [0.1]),
    (dict(TABLE, t_ref=0.0), [0.1]),
    (dict(TABLE, t_ref=np.nan), [0.1]),
    (dict(TABLE, p_ref=-1.0), [0.1]),
    (dict(TABLE, p_ref=np.inf), [0.1]),
    (TABLE, None),                                                 # fractions missing
    (TABLE, []),
    (TABLE, [[0.1, 0.2]]),
    (TABLE, [0.1, 1.5]),
    (TABLE, [-1e-9]),
    (TABLE, [np.nan]),
])
def test_continuum_args_rejects(table, x):
    with pytest.raises(ValueError):
        eng.continuum_args(table, x)
