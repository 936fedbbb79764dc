"""GPU tests of the solar beam (prb_set_solar_source -> k3_flux_solar and the solar passes of k3_flux_tma): totals, rows
and band fluxes against the FP64 restatement (tests/solar_flux_oracle.py) folded over the engine's own k matrix, the beam
alone, the exactness rules (no Sun, a dark Sun, rad_down_surface, eps = 1, one band, chunks), argument errors, the host
mirror (Atmosphere.columnFluxes) and the full-size cfg4 column under a blackbody Sun."""
import ctypes

import numpy as np
import pytest

from oracle import physics as ph
from pyrad_b200 import distributed as pd
from pyrad_b200 import engine as eng
from pyrad_b200 import workloads
from tests import flux_oracle as FO
from tests import solar_flux_oracle as SO
from tests.test_gpu_band_fluxes import RRTMG_LW, _column_on_data_tree, axis, band_floor, check_bands
from tests.test_gpu_flux_boundaries import CFG4_EPS, EPS_TABLES, small_edges
from tests.test_gpu_fluxes import (FLUX_FLOOR, FLUX_RTOL, ROWS_RTOL, data_root, device_kmatrix,  # noqa: F401
                                   pi_int_planck, quadrature, run_column, small_column)
from tests import helpers as H

pytestmark = pytest.mark.gpu

#: Sun tables on the small columns' 600-640 cm-1 axis, W m-2 (cm-1)-1: the beam is of the size of the thermal fluxes
#: there (pi B(288 K) ~ 0.35).  One covers the grid, one part of it, and a two-entry ramp.
SUNS = {"grid": ([590.0, 612.0, 627.0, 650.0], [0.25, 0.5, 0.15, 0.4]),
        "part": ([610.0, 618.0, 625.0], [0.4, 0.6, 0.2]),
        "ramp": ([605.0, 635.0], [0.0, 0.8])}
MU_SUNS = [1.0, 0.5, 0.05]
EPS_CASES = {"none": None, "constant": EPS_TABLES["constant"], "table": EPS_TABLES["table"]}
REFLECTIONS = ("lambertian", "specular")


@pytest.fixture()
def sengine(engine):
    """The session engine; its Sun and boundaries are cleared after the test."""
    try:
        yield engine
    finally:
        engine.set_solar_source()
        engine.set_flux_boundaries()


def blackbody_sun(nu_t, t_sun=5772.0, total=1361.0):
    """A blackbody Sun scaled to `total` W m-2 over all wavenumbers, as a table on nu_t (cm-1)."""
    fine = np.arange(1.0, 100000.0, 1.0)
    scale = total / (ph.pi * np.sum(ph.planck_wavenumber(fine, t_sun)))
    s = ph.pi * np.nan_to_num(ph.planck_wavenumber(np.asarray(nu_t, dtype=np.float64), t_sun)) * scale
    return np.asarray(nu_t, dtype=np.float64), s


def sun_floor(w, nu, sun, mu_sun, edges=None):
    """FLUX_FLOOR x mu_sun sum S res, in total or per band."""
    s = SO.irradiance(nu, sun) * mu_sun * w["res"] * FLUX_FLOOR
    if edges is None:
        return s.sum()
    idx = np.searchsorted(edges, nu, side="right") - 1
    sel = (idx >= 0) & (idx < len(edges) - 1)
    return np.bincount(idx[sel], weights=s[sel], minlength=len(edges) - 1)


def check_solar(w, got, ref, extra_floor):
    """check_fluxes with the floor raised by the Sun's share."""
    up, down, ru, rd = got
    r_up, r_down, r_ru, r_rd = ref
    ok = axis(w) > 0
    np.testing.assert_allclose(ru[:, ok], r_ru[:, ok], rtol=ROWS_RTOL)
    np.testing.assert_allclose(rd[:, ok], r_rd[:, ok], rtol=ROWS_RTOL)
    floor = FLUX_FLOOR * pi_int_planck(w) + extra_floor
    for a, b in ((up, r_up), (down, r_down)):
        err = np.abs(a - b)
        assert np.all(err <= FLUX_RTOL * np.abs(b) + floor), (err / np.maximum(np.abs(b), floor)).max()


def everything(engine, mu, wt, edges):
    return engine.atmosphere_fluxes(mu, wt, rows=True) + engine.atmosphere_band_fluxes(mu, wt, edges)


def assert_same_bits(a, b):
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


@pytest.mark.parametrize("L", [1, 3, 8, 24])
def test_solar_fluxes_match_the_fp64_fold_of_the_device_k_matrix(sengine, L):
    engine = sengine
    w = small_column(L)
    n = H.engine_setup(engine, w)
    run_column(engine, w)
    k = device_kmatrix(engine, L, n)
    nu = axis(w)
    edges = small_edges(nu)
    args = (k, w["depth_cm"], w["T"], w["t_surface"], nu, w["res"])
    for n_mu in (1, 2, 3, 4):
        mu, wt = quadrature(600 + L, n_mu)
        for reflection in REFLECTIONS:
            for j, eps in enumerate(EPS_CASES.values()):
                for m, sun in enumerate(SUNS.values()):
                    mu_sun = MU_SUNS[(n_mu + j + m) % 3]
                    t_top = 250.0 if (n_mu + m) % 3 == 0 else 0.0
                    engine.set_flux_boundaries(eps, reflection, t_top)
                    engine.set_solar_source(sun, mu_sun)
                    got = engine.atmosphere_fluxes(mu, wt, rows=True)
                    ref = SO.solar_fluxes(*args, mu, wt, sun, mu_sun, eps, reflection, t_top)
                    check_solar(w, got, ref, sun_floor(w, nu, sun, mu_sun))
                    if (n_mu + j + m) % 2 == 0:
                        bands = engine.atmosphere_band_fluxes(mu, wt, edges)
                        check_bands(bands, SO.solar_band_fluxes(*args, mu, wt, edges, sun, mu_sun, eps, reflection,
                                                                t_top),
                                    band_floor(w, nu, edges) + sun_floor(w, nu, sun, mu_sun, edges))


@pytest.mark.parametrize("mu_sun", MU_SUNS)
def test_the_beam_alone(sengine, mu_sun):
    """eps = 1, T_top = 0: the solar part of flux_down (Sun minus no Sun) is the oracle's beam term."""
    engine = sengine
    w = small_column(8)
    n = H.engine_setup(engine, w)
    run_column(engine, w)
    k = device_kmatrix(engine, 8, n)
    nu = axis(w)
    mu, wt = FO.gauss_legendre_01(3)
    for sun in SUNS.values():
        engine.set_solar_source()
        _, dark = engine.atmosphere_fluxes(mu, wt)
        engine.set_solar_source(sun, mu_sun)
        _, lit = engine.atmosphere_fluxes(mu, wt)
        ref = SO.beam_flux_down(k, w["depth_cm"], nu, w["res"], sun, mu_sun)
        np.testing.assert_allclose(lit - dark, ref, rtol=2e-5, atol=FLUX_FLOOR * pi_int_planck(w))
        assert ref[-1] > 0


@pytest.mark.parametrize("bounds", [None, (EPS_TABLES["table"], "specular", 250.0)])
def test_no_sun_set_and_a_cleared_sun_give_the_plain_bits(sengine, bounds):
    engine = sengine
    w = small_column(24)
    H.engine_setup(engine, w)
    run_column(engine, w)
    mu, wt = quadrature(8, 3)
    edges = small_edges(axis(w))
    engine.set_flux_boundaries(*(bounds or ()))
    never = everything(engine, mu, wt, edges)
    engine.set_solar_source(SUNS["grid"], 0.5)
    lit = everything(engine, mu, wt, edges)
    engine.set_solar_source()
    cleared = everything(engine, mu, wt, edges)
    assert_same_bits(never, cleared)
    assert not np.array_equal(lit[1], never[1]) and not np.array_equal(lit[5], never[5])


@pytest.mark.parametrize("bounds", [None, (None, "specular", 0.0), (EPS_TABLES["constant"], "lambertian", 0.0),
                                    (EPS_TABLES["table"], "lambertian", 250.0), (EPS_TABLES["table"], "specular", 2.725)])
def test_a_dark_sun_changes_nothing(sengine, bounds):
    engine = sengine
    w = small_column(8)
    H.engine_setup(engine, w)
    run_column(engine, w)
    edges = small_edges(axis(w))
    engine.set_flux_boundaries(*(bounds or ()))
    for n_mu in (1, 2, 4):
        mu, wt = quadrature(30 + n_mu, n_mu)
        engine.set_solar_source()
        ref = everything(engine, mu, wt, edges)
        for mu_sun in (1.0, 0.05):
            engine.set_solar_source(([590.0, 650.0], [0.0, 0.0]), mu_sun)
            assert_same_bits(everything(engine, mu, wt, edges), ref)


@pytest.mark.parametrize("reflection", REFLECTIONS)
def test_the_sun_never_changes_rad_down_surface(sengine, reflection):
    engine = sengine
    w = small_column(24)
    H.engine_setup(engine, w)
    run_column(engine, w)
    for n_mu in (1, 3, 4):
        mu, wt = quadrature(40 + n_mu, n_mu)
        for eps in EPS_CASES.values():
            engine.set_flux_boundaries(eps, reflection, 2.725)
            engine.set_solar_source()
            up, down, _, rd = engine.atmosphere_fluxes(mu, wt, rows=True)
            engine.set_solar_source(SUNS["part"], 0.5)
            up2, down2, _, rd2 = engine.atmosphere_fluxes(mu, wt, rows=True)
            assert rd2.tobytes() == rd.tobytes()
            # the beam only adds (it is exactly 0 at the levels it does not reach: this column absorbs all of it before
            # the lowest levels), and eps = 1 reflects nothing
            assert np.all(down2 >= down) and down2[-1] > down[-1]
            if eps is None:
                assert up2.tobytes() == up.tobytes()


@pytest.mark.parametrize("eps", [None, ([600.0, 620.0, 640.0], [1.0, 1.0, 1.0])])
def test_a_black_surface_reflects_no_sunlight(sengine, eps):
    engine = sengine
    w = small_column(8)
    H.engine_setup(engine, w)
    run_column(engine, w)
    edges = small_edges(axis(w))
    for n_mu in (1, 3, 4):
        mu, wt = quadrature(50 + n_mu, n_mu)
        for reflection in REFLECTIONS:
            engine.set_flux_boundaries(eps, reflection, 250.0)
            engine.set_solar_source()
            up, down, ru, _ = engine.atmosphere_fluxes(mu, wt, rows=True)
            bu, bd = engine.atmosphere_band_fluxes(mu, wt, edges)
            engine.set_solar_source(SUNS["grid"], 0.5)
            up2, down2, ru2, _ = engine.atmosphere_fluxes(mu, wt, rows=True)
            bu2, bd2 = engine.atmosphere_band_fluxes(mu, wt, edges)
            assert up2.tobytes() == up.tobytes() and ru2.tobytes() == ru.tobytes() and bu2.tobytes() == bu.tobytes()
            assert np.all(down2 >= down) and down2[-1] > down[-1] and np.all(bd2[:, -1] > bd[:, -1])


@pytest.mark.parametrize("L", [1, 3, 24])
def test_one_band_over_the_whole_axis_is_the_total_flux(sengine, L):
    engine = sengine
    w = small_column(L)
    H.engine_setup(engine, w)
    run_column(engine, w)
    for n_mu in (1, 2, 3, 4):
        mu, wt = quadrature(700 + L, n_mu)
        for reflection in REFLECTIONS:
            engine.set_flux_boundaries(EPS_TABLES["table"], reflection, 0.0)
            engine.set_solar_source(SUNS["part"], MU_SUNS[n_mu % 3])
            bu, bd = engine.atmosphere_band_fluxes(mu, wt, [w["range_min"], w["range_max"] + w["res"]])
            up, down = engine.atmosphere_fluxes(mu, wt)
            np.testing.assert_allclose(bu[0], up, rtol=1e-12, atol=0)
            np.testing.assert_allclose(bd[0], down, rtol=1e-12, atol=0)


@pytest.mark.parametrize("reflection", REFLECTIONS)
def test_chunks_give_the_same_rows_and_bands(sengine, reflection):
    """Two tile-aligned chunks on one engine: S and eps are resampled per chunk on the same axis, so the rows
    concatenate bit for bit, the totals add up, and a band inside one chunk gets the whole grid's bits."""
    engine = sengine
    w = small_column(24)
    n = H.engine_setup(engine, w)
    nu = axis(w)
    edges = np.array([nu[1000], nu[5000], nu[15000], nu[18000], nu[30000]])
    mu, wt = quadrature(5, 3)
    engine.set_flux_boundaries(EPS_TABLES["table"], reflection, 2.725)
    engine.set_solar_source(SUNS["grid"], 0.5)
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


def _set_raw(engine, nu, s, mu_sun):
    dp = ctypes.POINTER(ctypes.c_double)
    nu, s = np.ascontiguousarray(nu, dtype=np.float64), np.ascontiguousarray(s, dtype=np.float64)
    return engine._lib.prb_set_solar_source(engine._h, nu.size, nu.ctypes.data_as(dp) if nu.size else None,
                                            s.ctypes.data_as(dp) if s.size else None, mu_sun)


def test_argument_errors_keep_the_setting(sengine):
    engine = sengine
    w = small_column(3)
    H.engine_setup(engine, w)
    run_column(engine, w)
    mu, wt = quadrature(1, 2)
    engine.set_flux_boundaries(0.5, "specular", 0.0)
    engine.set_solar_source(SUNS["grid"], 0.5)
    good = engine.atmosphere_fluxes(mu, wt, rows=True)
    bad = [([600.0], [0.5], 0.5), ([600.0, 600.0], [0.5, 0.5], 0.5), ([610.0, 600.0], [0.5, 0.5], 0.5),
           ([600.0, np.nan], [0.5, 0.5], 0.5), ([-np.inf, 600.0], [0.5, 0.5], 0.5), ([600.0, 610.0], [0.5, -1e-9], 0.5),
           ([600.0, 610.0], [np.nan, 0.5], 0.5), ([600.0, 610.0], [0.5, np.inf], 0.5), ([600.0, 610.0], [0.5, 0.5], 0.0),
           ([600.0, 610.0], [0.5, 0.5], -0.5), ([600.0, 610.0], [0.5, 0.5], 1.5), ([600.0, 610.0], [0.5, 0.5], np.nan)]
    for args in bad:
        assert _set_raw(engine, *args) == -2, args                 # PRB_ERR_ARG
    dp = ctypes.POINTER(ctypes.c_double)
    two = np.array([0.5, 0.5])
    assert engine._lib.prb_set_solar_source(engine._h, 2, None, two.ctypes.data_as(dp), 0.5) == -2
    assert engine._lib.prb_set_solar_source(engine._h, 2, two.ctypes.data_as(dp), None, 0.5) == -2
    assert engine._lib.prb_set_solar_source(engine._h, -1, None, None, 0.5) == -2
    with pytest.raises(ValueError):
        engine.set_solar_source(SUNS["grid"], 0.0)
    again = engine.atmosphere_fluxes(mu, wt, rows=True)
    assert_same_bits(good, again)
    assert _set_raw(engine, [], [], np.nan) == 0                   # n_table = 0 clears; mu_sun is ignored
    plain = engine.atmosphere_fluxes(mu, wt, rows=True)
    engine.set_solar_source()
    assert_same_bits(plain, engine.atmosphere_fluxes(mu, wt, rows=True))
    assert plain[1][-1] == 0 and plain[1].tobytes() != good[1].tobytes()


def test_host_mirror_column_fluxes_with_a_sun(data_root, engine):
    """Atmosphere.columnFluxes(solarIrradiance=..., solarMu=...) gives the engine calls' bits, the heating rates follow
    the changed fluxes, and the Sun does not leak into the next call."""
    from pyrad_b200 import classes as C
    atm, rmin, rmax = _column_on_data_tree(data_root)
    mu, wt = FO.gauss_legendre_01(3)
    edges = np.linspace(rmin, rmax + 1.0, 5)
    sun = ([rmin - 1.0, 0.5 * (rmin + rmax), rmax + 1.0], [0.3, 0.6, 0.2])
    plain = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges)
    explicit = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges, solarIrradiance=None, solarMu=1.0)
    lit = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges, surfaceEmissivity=0.8, reflection="specular",
                           solarIrradiance=sun, solarMu=0.6)
    try:                                            # the engine still holds the column
        engine.set_flux_boundaries(0.8, "specular")
        engine.set_solar_source(sun, 0.6)
        up, down, ru, rd = engine.atmosphere_fluxes(mu, wt, rows=True)
        bu, bd = engine.atmosphere_band_fluxes(mu, wt, edges)
    finally:
        engine.set_solar_source()
        engine.set_flux_boundaries()
    for key, v in (("flux_up", up), ("flux_down", down), ("rad_up_top", ru), ("rad_down_surface", rd),
                   ("band_flux_up", bu), ("band_flux_down", bd)):
        np.testing.assert_array_equal(lit[key], v)
    after = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges)
    assert set(plain) == set(explicit) == set(lit) == set(after)
    for key in plain:
        np.testing.assert_array_equal(explicit[key], plain[key])
        np.testing.assert_array_equal(after[key], plain[key])
    assert np.all(lit["flux_down"] >= plain["flux_down"]) and lit["flux_down"][-1] > plain["flux_down"][-1]
    np.testing.assert_array_equal(lit["heating_rate"], C.heatingRate(lit["flux_up"], lit["flux_down"],
                                                                    [l.depth for l in atm], [l.T for l in atm],
                                                                    [l.P for l in atm]))
    with pytest.raises(ValueError, match="irradiance"):
        atm.columnFluxes(288, solarIrradiance=([rmax, rmin], [0.5, 0.5]))


def test_cfg4_full_size_solar_fluxes(sengine):
    """The 100-layer, 5 M-point cfg4 column with 3 Gauss-Legendre nodes, cfg4's surface (CFG4_EPS), the 2.725 K top and a
    5772 K blackbody Sun of 1361 W m-2 at mu_sun = 0.5, both reflections: level fluxes, and bands at RRTMG's 16
    longwave edges plus 2000, 4000, 4650 and 5000 + res cm-1, against the torch-FP64-on-device restatement of
    test_cfg4_full_size_boundary_fluxes extended with the beam (tests/solar_flux_oracle.py)."""
    import torch
    engine = sengine
    w = workloads.atmosphere()
    n = H.engine_setup(engine, w)
    L = len(w["T"])
    assert n == 5_000_000 and L == 100
    run_column(engine, w)
    mu, wt = FO.gauss_legendre_01(3)
    edges = np.array(sorted(set(RRTMG_LW) | {2000, 2600, 3250, 4000, 4650, w["range_max"] + w["res"]}), dtype=np.float64)
    nb = len(edges) - 1
    sun, mu_sun, t_top = blackbody_sun(np.arange(0.0, 5011.0)), 0.5, 2.725
    got = {}
    for reflection in REFLECTIONS:
        engine.set_flux_boundaries(CFG4_EPS, reflection, t_top)
        engine.set_solar_source(sun, mu_sun)
        got[reflection] = (engine.atmosphere_fluxes(mu, wt), engine.atmosphere_band_fluxes(mu, wt, edges))
    p, ld = engine.atmosphere_kmatrix_dev()
    kmat = pd.device_tensor(p, L * ld).view(L, ld)
    x0, dx, x_last, _ = eng.linspace_axis(w["range_min"], w["range_max"], n)
    h, c, kb = ph.h, ph.c, ph.k
    flt_max = float(np.finfo(np.float32).max)
    depth = [float(d) for d in w["depth_cm"]]
    r_tot = {r: torch.zeros(2, L + 1, dtype=torch.float64, device="cuda") for r in REFLECTIONS}
    r_band = {r: torch.zeros(2, nb + 1, L + 1, dtype=torch.float64, device="cuda") for r in REFLECTIONS}
    floor_b = torch.zeros(nb + 1, dtype=torch.float64, device="cuda")
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
            nu_np = nu.cpu().numpy()
            eps = torch.as_tensor(np.interp(nu_np, *CFG4_EPS).astype(np.float32), device="cuda").double()
            s_top = torch.as_tensor(SO.irradiance(nu_np, sun), device="cuda")
            floor_b.index_add_(0, ids, ph.pi * torch.nan_to_num(bs) + mu_sun * s_top)
            kneg[ids[(k < 0).any(dim=0)]] = True

            def level_add(r, d, j, f, I):
                I = torch.where(I.abs() <= flt_max, I, torch.zeros_like(I)) * f
                r_tot[r][d, j] += I.sum()
                r_band[r][d, :, j].index_add_(0, ids, I)

            def both(d, j, f, I):
                for r in REFLECTIONS:
                    level_add(r, d, j, f, I)

            rad_down, s = [], torch.zeros_like(nu)
            for m in range(3):
                f = 2 * ph.pi * wt[m] * mu[m] * w["res"]
                I = planck(t_top)
                both(1, L, f, I)
                for l in range(L - 1, -1, -1):
                    t = torch.exp(-k[l] * depth[l] / mu[m])
                    I = t * I + (1 - t) * B[l]
                    both(1, l, f, I)
                rad_down.append(I)
                s += 2 * wt[m] * mu[m] * I
            e = s_top
            both(1, L, mu_sun * w["res"], e)
            for l in range(L - 1, -1, -1):
                e = e * torch.exp(-k[l] * depth[l] / mu_sun)
                both(1, l, mu_sun * w["res"], e)
            for r in REFLECTIONS:
                for m in range(3):
                    f = 2 * ph.pi * wt[m] * mu[m] * w["res"]
                    sv = rad_down[m] if r == "specular" else s + mu_sun * e / ph.pi
                    I = torch.where(eps == 1, bs, eps * bs + (1 - eps) * sv)
                    level_add(r, 0, 0, f, I)
                    for l in range(L):
                        t = torch.exp(-k[l] * depth[l] / mu[m])
                        I = t * I + (1 - t) * B[l]
                        level_add(r, 0, l + 1, f, I)
                if r == "specular":
                    eu = torch.where(eps == 1, torch.zeros_like(e), (1 - eps) * e)
                    level_add(r, 0, 0, mu_sun * w["res"], eu)
                    for l in range(L):
                        eu = eu * torch.exp(-k[l] * depth[l] / mu_sun)
                        level_add(r, 0, l + 1, mu_sun * w["res"], eu)
    total_floor = FLUX_FLOOR * float(floor_b.sum()) * w["res"]
    floor = FLUX_FLOOR * floor_b[:-1].cpu().numpy() * w["res"]
    floor = np.where(kneg[:-1].cpu().numpy(), total_floor, floor)
    for r in REFLECTIONS:
        (up, down), bands = got[r]
        ref_up, ref_down = r_tot[r].cpu().numpy()
        for name, a_, b_ in (("up", up, ref_up), ("down", down, ref_down)):
            err = np.abs(a_ - b_) / np.maximum(np.abs(b_), total_floor)
            assert err.max() <= FLUX_RTOL, (r, name, err.max(), int(err.argmax()))
        check_bands(bands, [x[:-1].cpu().numpy() for x in r_band[r]], floor)
    # the beam brings ~80 W m-2 at the top (normal incidence; half of it on the level at mu_sun = 0.5)
    top_sun = mu_sun * np.sum(SO.irradiance(axis(w), sun)) * w["res"]
    assert 30 < top_sun < 50
    for r in REFLECTIONS:
        assert got[r][0][1][-1] == pytest.approx(top_sun, rel=1e-5)
