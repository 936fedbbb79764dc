"""CPU tests of the band-flux definitions (tests/band_flux_oracle.py): partitions add up to the column fluxes,
closed forms per band, band membership at and between grid values and outside the range, the band-edge validation of
Atmosphere.columnFluxes, and the rank-ordered sum of sharded band fluxes over a world-size-2 gloo run."""
import os
import socket

import numpy as np
import pytest

from oracle import physics as ph
from pyrad_b200 import classes as C
from pyrad_b200 import distributed as pd
from tests import band_flux_oracle as BO
from tests import flux_oracle as FO

RMIN, RMAX, RES = 0.0, 2500.0, 1.0          # includes the 0 cm-1 point, where Planck is 0/0 = NaN
NU = ph.x_axis(RMIN, RMAX, RES)
STEP = NU[1] - NU[0]


def random_column(L, seed, n=NU.size):
    rng = np.random.default_rng(seed)
    k = 10.0 ** rng.uniform(-8, 0, (L, n))
    depth = rng.uniform(1e4, 1e5, L)
    T = rng.uniform(200, 300, L)
    return k, depth, T


def pi_sum_planck(T, points):
    """pi sum_{points} B(nu, T) res, with the NaN of the 0 cm-1 point counted as 0."""
    return ph.pi * np.sum(np.nan_to_num(ph.planck_wavenumber(NU[points], T))) * RES


def transparent(edges, L=3, n_mu=3):
    mu, w = FO.gauss_legendre_01(n_mu)
    return BO.band_fluxes(np.zeros((L, NU.size)), np.full(L, 1e5), np.linspace(290, 210, L), 288.0, NU, RES, mu, w,
                          edges)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_bands_that_partition_the_axis_add_up_to_the_column_fluxes(seed):
    rng = np.random.default_rng(seed)
    k, depth, T = random_column(5, 10 + seed)
    mu, w = FO.gauss_legendre_01(1 + seed)
    inner = np.sort(rng.choice(NU[1:-1], 12, replace=False))
    inner[::3] += 0.4 * STEP                  # some edges between grid values
    edges = np.concatenate([[RMIN], inner, [RMAX + RES]])
    bu, bd = BO.band_fluxes(k, depth, T, 288.0, NU, RES, mu, w, edges)
    up, down, _, _ = FO.column_fluxes(k, depth, T, 288.0, NU, RES, mu, w)
    assert bu.shape == bd.shape == (13, 6)
    np.testing.assert_allclose(bu.sum(axis=0), up, rtol=1e-13)
    np.testing.assert_allclose(bd.sum(axis=0), down, rtol=1e-13)


def test_transparent_column_gives_pi_times_the_band_integral_of_the_surface():
    edges = np.array([0.0, 300.0, 667.5, 1000.0, 2500.0 + RES])
    bu, bd = transparent(edges)
    idx = np.searchsorted(edges, NU, side="right") - 1
    for b in range(4):
        np.testing.assert_allclose(bu[b], pi_sum_planck(288.0, idx == b), rtol=1e-12)
    assert np.all(bd == 0)


def test_isothermal_column_is_isotropic_per_band():
    k, depth, _ = random_column(6, 1)
    mu, w = FO.gauss_legendre_01(3)
    edges = np.array([10.0, 350.0, 500.0, 630.0, 700.0, 820.0, 980.0, 2000.0])
    bu, _ = BO.band_fluxes(k, depth, np.full(6, 250.0), 250.0, NU, RES, mu, w, edges)
    idx = np.searchsorted(edges, NU, side="right") - 1
    for b in range(7):
        np.testing.assert_allclose(bu[b], pi_sum_planck(250.0, idx == b), rtol=1e-12)


@pytest.mark.parametrize("edges,points", [
    ((NU[10], NU[20]), range(10, 20)),                              # on grid values: the lower edge's point is in
    ((NU[10] + 0.3 * STEP, NU[20] + 0.3 * STEP), range(11, 21)),    # between grid values
    ((-100.0, NU[5]), range(0, 5)),                                 # below range_min
    ((NU[-3], 1e6), range(NU.size - 3, NU.size)),                   # above range_max: the last point counts
    ((NU[-1], RMAX + RES), [NU.size - 1]),                          # the last point alone
    ((NU[7], NU[8]), [7]),                                          # a 1-point band
    ((NU[10] + 0.1 * STEP, NU[10] + 0.2 * STEP), []),               # a band between two points: empty
    ((RMAX + 1, RMAX + 2), []),                                     # wholly above the range: empty
])
def test_band_membership(edges, points):
    bu, bd = transparent(np.array(edges, dtype=np.float64))
    assert bu.shape == (1, 4)
    ref = pi_sum_planck(288.0, np.array(points, dtype=int))
    if points:
        np.testing.assert_allclose(bu[0], ref, rtol=1e-12)
    else:
        assert np.all(bu == 0)
    assert np.all(bd == 0)


def test_empty_bands_between_full_ones_give_zeros():
    edges = np.array([NU[3], NU[3] + 0.1 * STEP, NU[3] + 0.2 * STEP, NU[9], NU[9] + 0.5 * STEP])
    bu, _ = transparent(edges)
    np.testing.assert_allclose(bu[0], pi_sum_planck(288.0, [3]), rtol=1e-12)
    assert np.all(bu[1] == 0)
    np.testing.assert_allclose(bu[2], pi_sum_planck(288.0, range(4, 9)), rtol=1e-12)
    np.testing.assert_allclose(bu[3], pi_sum_planck(288.0, [9]), rtol=1e-12)


@pytest.mark.parametrize("bands", [
    [600.0], [], [[600.0, 700.0]], [700.0, 600.0], [600.0, 600.0], [600.0, np.nan], [600.0, np.inf], [-np.inf, 600.0],
])
def test_column_fluxes_rejects_bad_band_edges_before_the_column_runs(bands):
    atm = C.Atmosphere("empty")              # no layers: the column itself would fail, with another message
    with pytest.raises(ValueError, match="bands"):
        atm.columnFluxes(288.0, bands=bands)


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        k, depth, T = random_column(6, 5)
        mu, w = FO.gauss_legendre_01(3)
        edges = np.array([0.0, 350.0, 630.0, 700.0, 1023.5, 1800.0, 2080.0, 2500.0 + RES])
        cut = 1024                            # rank 0 owns [0, cut), rank 1 the rest; a band straddles the cut
        sl = slice(0, cut) if rank == 0 else slice(cut, NU.size)
        up, down = BO.band_fluxes(k[:, sl], depth, T, 288.0, NU[sl], RES, mu, w, edges)
        tot_up = pd.sum_over_ranks(up, dist)
        tot_down = pd.sum_over_ranks(down, dist)
        ref_up, ref_down = BO.band_fluxes(k, depth, T, 288.0, NU, RES, mu, w, edges)
        ok = (tot_up.shape == ref_up.shape == (7, 7) and np.allclose(tot_up, ref_up, rtol=1e-12, atol=0)
              and np.allclose(tot_down, ref_down, rtol=1e-12, atol=0))
        q.put((rank, bool(ok), tot_up.tobytes() + tot_down.tobytes()))
    finally:
        dist.destroy_process_group()


def test_sum_over_ranks_of_sharded_band_fluxes_equals_the_unsharded_band_fluxes():
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


def test_sum_over_ranks_without_a_process_group_keeps_a_2d_array():
    v = np.arange(12.0).reshape(3, 4)
    np.testing.assert_array_equal(pd.sum_over_ranks(v), v)
