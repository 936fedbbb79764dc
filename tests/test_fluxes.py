"""CPU tests of the column-flux definitions: the FP64 restatement (tests/flux_oracle.py) against closed forms, the
heating-rate formula of the host mirror, and the rank-ordered sum of sharded level fluxes over a world-size-2 gloo run."""
import os
import socket

import numpy as np
import pytest
from scipy.special import expn

from oracle import physics as ph
from pyrad_b200 import classes as C
from pyrad_b200 import distributed as pd
from tests import flux_oracle as FO

RMIN, RMAX, RES = 0.0, 2500.0, 1.0          # includes the 0 cm-1 point, where Planck is 0/0 = NaN
NU = ph.x_axis(RMIN, RMAX, RES)


def pi_int_planck(T, nu=NU):
    return ph.integrate_spectrum(ph.planck_wavenumber(nu, T), ph.pi, RES)


def random_column(L, seed, n=NU.size):
    rng = np.random.default_rng(seed)
    k = 10.0 ** rng.uniform(-8, 0, (L, n))
    depth = rng.uniform(1e4, 1e5, L)
    T = rng.uniform(200, 300, L)
    return k, depth, T


@pytest.mark.parametrize("n_mu", [1, 3, 4])
def test_transparent_column_carries_the_surface_up_and_nothing_down(n_mu):
    mu, w = FO.gauss_legendre_01(n_mu)
    L = 5
    up, down, ru, rd = FO.column_fluxes(np.zeros((L, NU.size)), np.full(L, 1e5), np.linspace(290, 210, L), 288.0, NU,
                                        RES, mu, w)
    np.testing.assert_allclose(up, pi_int_planck(288.0), rtol=1e-12)
    assert np.all(down == 0)
    assert ru.shape == rd.shape == (n_mu, NU.size) and np.isnan(ru[:, 0]).all() and np.all(rd[:, 1:] == 0)


def test_isothermal_column_at_the_surface_temperature_is_isotropic():
    k, depth, _ = random_column(6, 1)
    mu, w = FO.gauss_legendre_01(3)
    up, _, _, _ = FO.column_fluxes(k, depth, np.full(6, 250.0), 250.0, NU, RES, mu, w)
    np.testing.assert_allclose(up, pi_int_planck(250.0), rtol=1e-12)


def test_opaque_bottom_layer_sends_its_own_emission_down():
    k, depth, T = random_column(4, 2)
    k[0] = 1.0                                # tau = depth >= 1e4: T = 0 exactly
    mu, w = FO.gauss_legendre_01(3)
    _, down, _, rd = FO.column_fluxes(k, depth, T, 288.0, NU, RES, mu, w)
    np.testing.assert_allclose(down[0], pi_int_planck(T[0]), rtol=1e-12)
    np.testing.assert_array_equal(rd[:, 1:], np.broadcast_to(ph.planck_wavenumber(NU, T[0])[1:], (3, NU.size - 1)))


@pytest.mark.parametrize("tau", [0.1, 0.3, 1.0, 3.0])
def test_gray_cold_layer_gives_the_exponential_integral(tau):
    """F_up at the top of one gray layer of optical depth tau that emits nothing is pi B(T_s) 2 E3(tau): pins the
    angular convention (2 pi sum w mu, T = exp(-tau / mu)).  (Below tau ~ 0.05 the integrand mu exp(-tau / mu) turns
    sharply near mu ~ tau and the 16-node rule itself misses 2 E3 by more than 1e-6.)"""
    nu = ph.x_axis(500.0, 1500.0, RES)
    assert np.all(ph.planck_wavenumber(nu, 1.0) == 0)
    mu, w = FO.gauss_legendre_01(16)
    depth = 1e3
    up, down, _, _ = FO.column_fluxes([np.full(nu.size, tau / depth)], [depth], [1.0], 288.0, nu, RES, mu, w)
    ref = ph.integrate_spectrum(ph.planck_wavenumber(nu, 288.0), ph.pi, RES) * 2 * expn(3, tau)
    assert up[1] == pytest.approx(ref, rel=1e-6)
    assert np.all(down == 0)


def test_one_vertical_node_is_the_layer_by_layer_transmission_chain():
    k, depth, T = random_column(7, 3)
    _, _, ru, _ = FO.column_fluxes(k, depth, T, 288.0, NU, RES, [1.0], [0.5])
    I = ph.planck_wavenumber(NU, 288.0)
    for l in range(7):
        I = ph.transmission(ph.transmittance(k[l], depth[l]), I, ph.planck_wavenumber(NU, T[l]))
    np.testing.assert_array_equal(ru[0], I)
    # and F_up at the top is integrateSpectrum of the nadir radiance with the pi of the plotSpectrum legend
    up, _, _, _ = FO.column_fluxes(k, depth, T, 288.0, NU, RES, [1.0], [0.5])
    assert up[-1] == pytest.approx(ph.integrate_spectrum(I, ph.pi, RES), rel=1e-13)


def test_heating_rate_by_hand():
    up = np.array([400.0, 390.0, 385.0])
    down = np.array([300.0, 200.0, 0.0])
    depth, T, P = [1e5, 2e5], [280.0, 250.0], [900.0, 500.0]
    q = C.heatingRate(up, down, depth, T, P)
    net = up - down                           # 100, 190, 385
    rho = [100 * 900.0 * 0.0289647 / (8.314462618 * 280.0), 100 * 500.0 * 0.0289647 / (8.314462618 * 250.0)]
    ref = [-(190 - 100) / (rho[0] * 1004.64 * 1000.0) * 86400, -(385 - 190) / (rho[1] * 1004.64 * 2000.0) * 86400]
    np.testing.assert_allclose(q, ref, rtol=1e-14)
    assert q[0] == pytest.approx(-6.913, abs=1e-3)         # 90 W m-2 out of 1 km of air at 900 hPa, 280 K (1.12 kg m-3)
    with pytest.raises(ValueError):
        C.heatingRate(up[:2], down[:2], depth, T, P)


def test_top_of_an_isothermal_column_cools():
    k, depth, _ = random_column(5, 4)
    T = np.full(5, 260.0)
    mu, w = FO.gauss_legendre_01(3)
    up, down, _, _ = FO.column_fluxes(k, depth, T, 260.0, NU, RES, mu, w)
    q = C.heatingRate(up, down, depth, T, np.geomspace(1000.0, 10.0, 5))
    assert q[-1] < 0


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        k, depth, T = random_column(6, 5)
        mu, w = FO.gauss_legendre_01(3)
        cut = 1024 * 1                        # rank 0 owns [0, cut), rank 1 the rest
        sl = slice(0, cut) if rank == 0 else slice(cut, NU.size)
        up, down, _, _ = FO.column_fluxes(k[:, sl], depth, T, 288.0, NU[sl], RES, mu, w)
        tot_up = pd.sum_over_ranks(up, dist)
        tot_down = pd.sum_over_ranks(down, dist)
        ref_up, ref_down, _, _ = FO.column_fluxes(k, depth, T, 288.0, NU, RES, mu, w)
        ok = np.allclose(tot_up, ref_up, rtol=1e-12, atol=0) and np.allclose(tot_down, ref_down, rtol=1e-12, atol=0)
        q.put((rank, bool(ok), tot_up.tobytes() + tot_down.tobytes()))
    finally:
        dist.destroy_process_group()


def test_sum_over_ranks_of_sharded_fluxes_equals_the_unsharded_fluxes():
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(ok for _, ok, _ in res), res
    assert res[0][2] == res[1][2]             # every rank holds the same bits


def test_sum_over_ranks_without_a_process_group_is_the_identity():
    v = np.array([1.0, 2.5, -3.0])
    np.testing.assert_array_equal(pd.sum_over_ranks(v), v)
