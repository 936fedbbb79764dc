"""GPU tests of the flux boundaries (prb_set_flux_boundaries -> k3_flux_emissivity and the boundary passes of
k3_flux_tma): totals, rows and band fluxes against the FP64 restatement (tests/boundary_flux_oracle.py) folded over the
engine's own k matrix, the exactness rules (eps = 1 and T_top = 0 change nothing, bit for bit), the isothermal closed
form, the one-band identity, chunk invariance, argument errors, the host mirror (Atmosphere.columnFluxes) and the
full-size cfg4 column."""
import ctypes

import numpy as np
import pytest

from oracle import physics as ph
from pyrad_b200 import distributed as pd
from pyrad_b200 import engine as eng
from pyrad_b200 import workloads
from tests import boundary_flux_oracle as XO
from tests import flux_oracle as FO
from tests import helpers as H
from tests.test_gpu_band_fluxes import RRTMG_LW, _column_on_data_tree, axis, band_floor, check_bands
from tests.test_gpu_fluxes import (FLUX_FLOOR, FLUX_RTOL, check_fluxes, data_root, device_kmatrix,  # noqa: F401
                                   quadrature, run_column, small_column)

pytestmark = pytest.mark.gpu

#: emissivity tables on the small columns' 600-640 cm-1 axis: a constant, a table that reaches 0 and 1 inside the
#: grid, and a one-entry table
EPS_TABLES = {"constant": 0.9,
              "table": ([595.0, 605.0, 612.0, 620.0, 626.5, 633.0, 650.0], [0.6, 1.0, 1.0, 0.0, 0.35, 0.8, 0.5]),
              "one_entry": ([615.0], [0.7])}
T_TOPS = [0.0, 2.725, 250.0]
#: cfg4's surface: 0.98 with a linear dip to 0.75 over 1080-1180 cm-1
CFG4_EPS = ([1080.0, 1130.0, 1180.0], [0.98, 0.75, 0.98])


@pytest.fixture()
def bengine(engine):
    """The session engine; its boundaries are cleared after the test."""
    try:
        yield engine
    finally:
        engine.set_flux_boundaries()


def small_edges(nu):
    step = nu[1] - nu[0]
    return np.array([nu[0], nu[100], nu[128] + 0.5 * step, nu[1024], nu[9000], nu[20000], nu[-1] - 3.0, nu[-1] + step])


@pytest.mark.parametrize("L", [1, 3, 8, 24])
def test_boundary_fluxes_match_the_fp64_fold_of_the_device_k_matrix(bengine, L):
    engine = bengine
    w = small_column(L)
    n = H.engine_setup(engine, w)
    run_column(engine, w)
    k = device_kmatrix(engine, L, n)
    nu = axis(w)
    edges = small_edges(nu)
    floor = band_floor(w, nu, edges)
    args = (k, w["depth_cm"], w["T"], w["t_surface"], nu, w["res"])
    for n_mu in (1, 2, 3, 4):
        mu, wt = quadrature(400 + L, n_mu)
        for reflection in ("lambertian", "specular"):
            for j, (name, eps) in enumerate(EPS_TABLES.items()):
                for t_top in T_TOPS:
                    engine.set_flux_boundaries(eps, reflection, t_top)
                    got = engine.atmosphere_fluxes(mu, wt, rows=True)
                    ref = XO.boundary_fluxes(*args, mu, wt, eps, reflection, t_top)
                    check_fluxes(w, got, ref)
                    if (n_mu + j) % 2 == 0 or t_top == 2.725:
                        bands = engine.atmosphere_band_fluxes(mu, wt, edges)
                        check_bands(bands, XO.boundary_band_fluxes(*args, mu, wt, edges, eps, reflection, t_top), floor)
                    if t_top != 2.725:                        # (B(nu, 2.725 K) underflows FP32 at 600 cm-1)
                        assert (got[1][-1] == 0) == (t_top == 0), (name, reflection, t_top)


def test_set_then_cleared_equals_never_set(bengine):
    engine = bengine
    w = small_column(24)
    H.engine_setup(engine, w)
    run_column(engine, w)
    mu, wt = quadrature(8, 3)
    edges = small_edges(axis(w))
    before = engine.atmosphere_fluxes(mu, wt, rows=True) + engine.atmosphere_band_fluxes(mu, wt, edges)
    engine.set_flux_boundaries(EPS_TABLES["table"], "specular", 250.0)
    grey = engine.atmosphere_fluxes(mu, wt, rows=True)
    engine.set_flux_boundaries()
    after = engine.atmosphere_fluxes(mu, wt, rows=True) + engine.atmosphere_band_fluxes(mu, wt, edges)
    for a, b in zip(before, after):
        assert a.tobytes() == b.tobytes()
    assert not np.array_equal(grey[0], before[0]) and not np.array_equal(grey[1], before[1])


@pytest.mark.parametrize("eps", [None, 1.0, ([600.0, 620.0, 640.0], [1.0, 1.0, 1.0])])
def test_a_black_surface_under_a_warm_top_leaves_the_upward_results_alone(bengine, eps):
    engine = bengine
    w = small_column(8)
    H.engine_setup(engine, w)
    run_column(engine, w)
    edges = small_edges(axis(w))
    for n_mu in (1, 3, 4):
        mu, wt = quadrature(9 + n_mu, n_mu)
        engine.set_flux_boundaries()
        up, down, ru, rd = engine.atmosphere_fluxes(mu, wt, rows=True)
        bu, bd = engine.atmosphere_band_fluxes(mu, wt, edges)
        for reflection in ("lambertian", "specular"):
            engine.set_flux_boundaries(eps, reflection, 250.0)
            up2, down2, ru2, rd2 = engine.atmosphere_fluxes(mu, wt, rows=True)
            bu2, bd2 = engine.atmosphere_band_fluxes(mu, wt, edges)
            assert up2.tobytes() == up.tobytes() and ru2.tobytes() == ru.tobytes() and bu2.tobytes() == bu.tobytes()
            assert down[-1] == 0 and down2[-1] > 0 and np.all(bd2[:, -1] > 0)


@pytest.mark.parametrize("name", list(EPS_TABLES))
def test_a_cold_top_leaves_the_downward_results_alone(bengine, name):
    engine = bengine
    w = small_column(24)
    H.engine_setup(engine, w)
    run_column(engine, w)
    edges = small_edges(axis(w))
    for n_mu in (2, 3):
        mu, wt = quadrature(20 + n_mu, n_mu)
        engine.set_flux_boundaries()
        up, down, ru, rd = engine.atmosphere_fluxes(mu, wt, rows=True)
        bu, bd = engine.atmosphere_band_fluxes(mu, wt, edges)
        for reflection in ("lambertian", "specular"):
            engine.set_flux_boundaries(EPS_TABLES[name], reflection, 0.0)
            up2, down2, ru2, rd2 = engine.atmosphere_fluxes(mu, wt, rows=True)
            bu2, bd2 = engine.atmosphere_band_fluxes(mu, wt, edges)
            assert down2.tobytes() == down.tobytes() and rd2.tobytes() == rd.tobytes() and bd2.tobytes() == bd.tobytes()
            assert up2[0] != up[0]                                    # the surface itself did change


@pytest.mark.parametrize("reflection", ["lambertian", "specular"])
def test_isothermal_column_under_an_isothermal_top_is_isotropic(bengine, reflection):
    engine = bengine
    w = dict(small_column(8))
    L = len(w["T"])
    w["T"] = [250.0] * L
    w["t_surface"] = 250.0
    n = H.engine_setup(engine, w)
    run_column(engine, w)
    nu = axis(w)
    b = ph.planck_wavenumber(nu, 250.0)
    ref = ph.integrate_spectrum(b, ph.pi, w["res"])
    for n_mu in (1, 3, 4):
        mu, wt = FO.gauss_legendre_01(n_mu)
        engine.set_flux_boundaries(EPS_TABLES["table"], reflection, 250.0)
        up, down, ru, rd = engine.atmosphere_fluxes(mu, wt, rows=True)
        np.testing.assert_allclose(up, ref, rtol=1e-6)
        np.testing.assert_allclose(down, ref, rtol=1e-6)
        for rows in (ru, rd):
            np.testing.assert_allclose(rows, np.broadcast_to(b, (n_mu, n)), rtol=1e-6)


@pytest.mark.parametrize("L", [1, 3, 24])
def test_one_band_over_the_whole_axis_is_the_total_flux(bengine, L):
    engine = bengine
    w = small_column(L)
    H.engine_setup(engine, w)
    run_column(engine, w)
    for n_mu in (1, 2, 3, 4):
        mu, wt = quadrature(500 + L, n_mu)
        for reflection in ("lambertian", "specular"):
            engine.set_flux_boundaries(EPS_TABLES["table"], reflection, 250.0)
            bu, bd = engine.atmosphere_band_fluxes(mu, wt, [w["range_min"], w["range_max"] + w["res"]])
            up, down = engine.atmosphere_fluxes(mu, wt)
            np.testing.assert_allclose(bu[0], up, rtol=1e-12, atol=0)
            np.testing.assert_allclose(bd[0], down, rtol=1e-12, atol=0)


def test_chunks_give_the_same_rows_and_bands(bengine):
    """Two tile-aligned chunks on one engine: the emissivity is resampled per chunk on the same axis, so the rows
    concatenate bit for bit, the totals add up, and a band inside one chunk gets the whole grid's bits."""
    engine = bengine
    w = small_column(24)
    n = H.engine_setup(engine, w)
    nu = axis(w)
    edges = np.array([nu[1000], nu[5000], nu[15000], nu[18000], nu[30000]])
    mu, wt = quadrature(5, 3)
    engine.set_flux_boundaries(EPS_TABLES["table"], "lambertian", 2.725)
    run_column(engine, w)
    full = engine.atmosphere_fluxes(mu, wt, rows=True)
    full_b = engine.atmosphere_band_fluxes(mu, wt, edges)
    parts, parts_b = [], []
    for a, b in ((0, 16384), (16384, n)):
        H.engine_setup(engine, w, a, b)
        run_column(engine, w)
        parts.append(engine.atmosphere_fluxes(mu, wt, rows=True))
        parts_b.append(engine.atmosphere_band_fluxes(mu, wt, edges))
    for r in (2, 3):
        np.testing.assert_array_equal(np.concatenate([p[r] for p in parts], axis=1), full[r])
    for f in (0, 1):
        np.testing.assert_allclose(parts[0][f] + parts[1][f], full[f], rtol=1e-12, atol=0)
        np.testing.assert_array_equal(parts_b[0][f][0], full_b[f][0])          # [nu_1000, nu_5000)
        np.testing.assert_array_equal(parts_b[1][f][3], full_b[f][3])          # [nu_18000, nu_30000)
        np.testing.assert_allclose(parts_b[0][f][2] + parts_b[1][f][2], full_b[f][2], rtol=1e-12, atol=0)


def _set_raw(engine, nu, eps, reflection, t_top):
    dp = ctypes.POINTER(ctypes.c_double)
    nu, eps = np.ascontiguousarray(nu, dtype=np.float64), np.ascontiguousarray(eps, dtype=np.float64)
    return engine._lib.prb_set_flux_boundaries(engine._h, nu.size, nu.ctypes.data_as(dp) if nu.size else None,
                                               eps.ctypes.data_as(dp) if eps.size else None, reflection, t_top)


def test_argument_errors_keep_the_setting(bengine):
    engine = bengine
    w = small_column(3)
    H.engine_setup(engine, w)
    run_column(engine, w)
    mu, wt = quadrature(1, 2)
    engine.set_flux_boundaries(EPS_TABLES["table"], "specular", 250.0)
    good = engine.atmosphere_fluxes(mu, wt, rows=True)
    bad = [([600.0, 600.0], [0.5, 0.5], 0, 0.0), ([610.0, 600.0], [0.5, 0.5], 0, 0.0),
           ([600.0, np.nan], [0.5, 0.5], 0, 0.0), ([-np.inf, 600.0], [0.5, 0.5], 0, 0.0),
           ([600.0], [1.5], 0, 0.0), ([600.0], [-0.01], 0, 0.0), ([600.0], [np.nan], 0, 0.0),
           ([600.0], [0.5], 2, 0.0), ([600.0], [0.5], -1, 0.0), ([], [], 0, -1.0), ([], [], 0, np.inf),
           ([], [], 0, np.nan)]
    for args in bad:
        assert _set_raw(engine, *args) == -2, args                 # PRB_ERR_ARG
    dp = ctypes.POINTER(ctypes.c_double)
    one = np.array([0.5])
    assert engine._lib.prb_set_flux_boundaries(engine._h, 1, None, one.ctypes.data_as(dp), 0, 0.0) == -2
    assert engine._lib.prb_set_flux_boundaries(engine._h, -1, None, None, 0, 0.0) == -2
    with pytest.raises(ValueError):
        engine.set_flux_boundaries(1.5)
    again = engine.atmosphere_fluxes(mu, wt, rows=True)
    for a, b in zip(good, again):
        assert a.tobytes() == b.tobytes()
    assert _set_raw(engine, [], [], 0, 0.0) == 0                   # (0, NULL, NULL, 0, 0.0): the defaults
    engine.set_flux_boundaries()
    plain = engine.atmosphere_fluxes(mu, wt, rows=True)
    assert plain[1][-1] == 0 and plain[0].tobytes() != good[0].tobytes()


def test_host_mirror_column_fluxes_with_boundaries(data_root):
    """Atmosphere.columnFluxes on the data-tree column: the default boundaries give the plain result bit for bit, a call
    with a surface does not leak into the next call, and the heating rates follow the changed fluxes."""
    from pyrad_b200 import classes as C
    atm, rmin, rmax = _column_on_data_tree(data_root)
    mu, wt = FO.gauss_legendre_01(3)
    edges = np.linspace(rmin, rmax + 1.0, 5)
    plain = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges)
    explicit = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges, surfaceEmissivity=None, reflection="lambertian",
                                topTemperature=0.0)
    grey = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges, surfaceEmissivity=0.8, reflection="lambertian",
                            topTemperature=2.725)
    after = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges)
    assert set(plain) == set(explicit) == set(grey) == set(after)
    for key in plain:
        np.testing.assert_array_equal(explicit[key], plain[key])
        np.testing.assert_array_equal(after[key], plain[key])
    # a grey surface under a colder sky emits less and loses less net flux; this column is opaque at every point
    # within FP32, so the top does not see it
    assert grey["flux_up"][0] < plain["flux_up"][0] and grey["net"][0] < plain["net"][0]
    assert grey["flux_up"][-1] <= plain["flux_up"][-1]
    np.testing.assert_array_equal(grey["heating_rate"], C.heatingRate(grey["flux_up"], grey["flux_down"],
                                                                      [l.depth for l in atm], [l.T for l in atm],
                                                                      [l.P for l in atm]))
    with pytest.raises(ValueError, match="emissivity"):
        atm.columnFluxes(288, surfaceEmissivity=([rmax, rmin], [0.5, 0.5]))


def test_cfg4_full_size_boundary_fluxes(bengine):
    """The 100-layer, 5 M-point cfg4 column with 3 Gauss-Legendre nodes, a surface of emissivity 0.98 with a linear dip
    to 0.75 over 1080-1180 cm-1, Lambertian, under the 2.725 K cosmic background: level fluxes and RRTMG's 16 longwave
    bands against the torch-FP64-on-device restatement of test_cfg4_full_size_band_fluxes with the boundaries of
    tests/boundary_flux_oracle.py (downward pass first, eps np.interp rounded to FP32)."""
    import torch
    engine = bengine
    w = workloads.atmosphere()
    n = H.engine_setup(engine, w)
    L = len(w["T"])
    assert n == 5_000_000 and L == 100
    run_column(engine, w)
    mu, wt = FO.gauss_legendre_01(3)
    edges = np.array(RRTMG_LW, dtype=np.float64)
    nb = len(edges) - 1
    plain = engine.atmosphere_fluxes(mu, wt)
    engine.set_flux_boundaries(CFG4_EPS, "lambertian", 2.725)
    up, down = engine.atmosphere_fluxes(mu, wt)
    bu, bd = engine.atmosphere_band_fluxes(mu, wt, edges)
    p, ld = engine.atmosphere_kmatrix_dev()
    kmat = pd.device_tensor(p, L * ld).view(L, ld)
    x0, dx, x_last, _ = eng.linspace_axis(w["range_min"], w["range_max"], n)
    h, c, kb = ph.h, ph.c, ph.k
    flt_max = float(np.finfo(np.float32).max)
    depth = [float(d) for d in w["depth_cm"]]
    r_tot = torch.zeros(2, L + 1, dtype=torch.float64, device="cuda")
    r_band = torch.zeros(2, nb + 1, L + 1, dtype=torch.float64, device="cuda")
    pib = torch.zeros(nb + 1, dtype=torch.float64, device="cuda")
    kneg = torch.zeros(nb + 1, dtype=torch.bool, device="cuda")
    edges_t = torch.as_tensor(edges, device="cuda")
    block = 1 << 20
    with torch.no_grad():
        for a in range(0, n, block):
            b = min(n, a + block)
            nu = torch.arange(a, b, dtype=torch.float64, device="cuda") * dx + x0
            if b == n:
                nu[-1] = x_last

            def planck(T):
                return 2E8 * h * c ** 2 * nu ** 3 / (torch.exp(100 * h * c * nu / kb / float(T)) - 1)

            i = torch.searchsorted(edges_t, nu, right=True) - 1
            ids = torch.where((i >= 0) & (i < nb), i, torch.full_like(i, nb))
            B = [planck(T) for T in w["T"]]
            k = kmat[:, a:b].double()
            bs = planck(w["t_surface"])
            pib.index_add_(0, ids, torch.nan_to_num(bs))
            kneg[ids[(k < 0).any(dim=0)]] = True
            eps = torch.as_tensor(np.interp(nu.cpu().numpy(), *CFG4_EPS).astype(np.float32), device="cuda").double()

            def level_add(d, j, f, I):
                I = torch.where(I.abs() <= flt_max, I, torch.zeros_like(I)) * f
                r_tot[d, j] += I.sum()
                r_band[d, :, j].index_add_(0, ids, I)

            s = torch.zeros_like(nu)
            for m in range(3):
                f = 2 * ph.pi * wt[m] * mu[m] * w["res"]
                I = planck(2.725)
                level_add(1, L, f, I)
                for l in range(L - 1, -1, -1):
                    t = torch.exp(-k[l] * depth[l] / mu[m])
                    I = t * I + (1 - t) * B[l]
                    level_add(1, l, f, I)
                s += 2 * wt[m] * mu[m] * I
            for m in range(3):
                f = 2 * ph.pi * wt[m] * mu[m] * w["res"]
                I = torch.where(eps == 1, bs, eps * bs + (1 - eps) * s)
                level_add(0, 0, f, I)
                for l in range(L):
                    t = torch.exp(-k[l] * depth[l] / mu[m])
                    I = t * I + (1 - t) * B[l]
                    level_add(0, l + 1, f, I)
    total_floor = FLUX_FLOOR * ph.integrate_spectrum(
        ph.planck_wavenumber(ph.x_axis(w["range_min"], w["range_max"], w["res"]), w["t_surface"]), ph.pi, w["res"])
    ref_up, ref_down = r_tot.cpu().numpy()
    for name, a_, b_ in (("up", up, ref_up), ("down", down, ref_down)):
        err = np.abs(a_ - b_) / np.maximum(np.abs(b_), total_floor)
        assert err.max() <= FLUX_RTOL, (name, err.max(), int(err.argmax()), a_[int(err.argmax())], b_[int(err.argmax())])
    floor = FLUX_FLOOR * ph.pi * pib[:-1].cpu().numpy() * w["res"]
    floor = np.where(kneg[:-1].cpu().numpy(), total_floor, floor)
    check_bands((bu, bd), [r[:-1].cpu().numpy() for r in r_band], floor)
    # the grey surface emits less and so loses less net flux; the cosmic background adds ~3e-6 W m-2 at the top.  (The
    # OLR does not move: no surface radiation gets through this column's 5 M lines within FP32.)
    assert up[0] < plain[0][0] and up[0] - down[0] < plain[0][0] - plain[1][0] and 0 < down[-1] < 1e-3
    assert up[-1] <= plain[0][-1]
