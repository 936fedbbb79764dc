"""GPU tests of the water-vapour continuum (prb_set_continuum -> k3_continuum_rows, k3_continuum_add): the k matrix
against the FP64 restatement (tests/continuum_oracle.py) added to the same column's k matrix without it, the column's
radiance and transmittance over both folds, fluxes and band fluxes, the exactness rules, the gas cell, chunks, argument
and state errors, the host mirror (Atmosphere.columnFluxes) and the full-size cfg4 column."""
import ctypes

import numpy as np
import pytest

from oracle import physics as ph
from pyrad_b200 import _lib
from pyrad_b200 import distributed as pd
from pyrad_b200 import engine as eng
from pyrad_b200 import workloads
from tests import band_flux_oracle as BO
from tests import continuum_oracle as CO
from tests import flux_oracle as FO
from tests import helpers as H
from tests import solar_flux_oracle as SO
from tests.test_gpu_band_fluxes import _column_on_data_tree, axis, band_floor, check_bands
from tests.test_gpu_flux_boundaries import EPS_TABLES, small_edges
from tests.test_gpu_fluxes import (data_root, device_kmatrix, quadrature, run_column, small_column,  # noqa: F401
                                   check_fluxes)
from tests.test_gpu_solar_flux import SUNS, check_solar, sun_floor

pytestmark = pytest.mark.gpu

KC_RTOL = 2e-6                  # of k_c, plus one FP32 ulp of k + k_c


@pytest.fixture()
def cengine(engine):
    """The session engine; its continuum, Sun and boundaries are cleared after the test."""
    try:
        yield engine
    finally:
        engine.set_continuum()
        engine.set_solar_source()
        engine.set_flux_boundaries()
        engine.set_option(eng.OPT_FOLD_TMA, 1)


def small_table(seed):
    """A synthetic table over the small columns' 600-640 cm-1 axis and beyond it, ~10 cm-1 apart."""
    return CO.synthetic_table(seed, 590.0, 650.0)


def kmatrix_f32(engine, L, n):
    import torch
    p, ld = engine.atmosphere_kmatrix_dev()
    k = pd.device_tensor(p, L * ld).view(L, ld)[:, :n]
    torch.cuda.synchronize()
    return k.cpu().numpy().copy()


def check_kmatrix(k_dev, k_lines, kc):
    """|k_dev - (k_lines + k_c)| <= KC_RTOL k_c + one FP32 ulp of the sum."""
    ref = k_lines.astype(np.float64) + kc
    ulp = np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
    err = np.abs(k_dev.astype(np.float64) - ref)
    bad = err > KC_RTOL * np.abs(kc) + ulp
    assert not bad.any(), (int(bad.sum()), float((err / np.maximum(np.abs(kc), 1e-300)).max()))


def fold_fp64(k, w):
    """The column's nadir radiance and total transmittance in FP64 (the reference's layer step, upward)."""
    nu = axis(w)
    I = ph.planck_wavenumber(nu, w["t_surface"])
    tt = np.ones_like(nu)
    for l in range(len(w["T"])):
        t = np.exp(-np.asarray(k[l], dtype=np.float64) * w["depth_cm"][l])
        I = ph.transmission(t, I, ph.planck_wavenumber(nu, w["T"][l]))
        tt = tt * t
    return I, tt


def read_f32(engine):
    rad = np.empty(engine.n_chunk, dtype=np.float32)
    tr = np.empty(engine.n_chunk, dtype=np.float32)
    engine.atmosphere_read_f32(rad, tr)
    return rad, tr


def lines_and_continuum(engine, w, table, x):
    """The column's device k matrix without a continuum, then with it (the engine keeps the second)."""
    L = len(w["T"])
    n = H.engine_setup(engine, w)
    engine.set_continuum()
    run_column(engine, w)
    k_lines = kmatrix_f32(engine, L, n)
    engine.set_continuum(table, x)
    run_column(engine, w)
    return k_lines, kmatrix_f32(engine, L, n)


@pytest.mark.parametrize("L", [1, 3, 8, 24])
def test_kmatrix_is_the_lines_plus_the_oracle_continuum(cengine, L):
    engine = cengine
    w = small_column(L)
    table, x = small_table(L), CO.synthetic_mole_fractions(L, L)
    k_lines, k_dev = lines_and_continuum(engine, w, table, x)
    kc = CO.continuum(axis(w), w["T"], w["P"], x, table)
    assert np.all(kc[:, axis(w) > 0] > 0)
    check_kmatrix(k_dev, k_lines, kc)


@pytest.mark.parametrize("L,tma", [(1, 1), (3, 1), (8, 1), (8, 0), (24, 1), (24, 0)])
def test_radiance_and_transmittance_match_the_fp64_fold(cengine, L, tma):
    engine = cengine
    w = small_column(L)
    n = H.engine_setup(engine, w)
    engine.set_option(eng.OPT_FOLD_TMA, tma)
    engine.set_continuum(small_table(7 + L), CO.synthetic_mole_fractions(7 + L, L))
    run_column(engine, w)
    if L == 1:
        assert engine.atmosphere_launches() >= 4          # K1, K2, the add and k3_fold_f32 (no fused epilogue)
    k = device_kmatrix(engine, L, n)
    rad, tr = read_f32(engine)
    I, tt = fold_fp64(k, w)
    ok = axis(w) > 0
    np.testing.assert_allclose(rad[ok], I[ok], rtol=2e-5)
    assert np.abs(tr - tt).max() <= H.T_ABS_TOL


@pytest.mark.parametrize("L", [1, 3, 8, 24])
def test_fluxes_and_bands_match_the_oracle_on_k_plus_kc(cengine, L):
    engine = cengine
    w = small_column(L)
    table, x = small_table(20 + L), CO.synthetic_mole_fractions(20 + L, L)
    k_lines, _ = lines_and_continuum(engine, w, table, x)
    nu = axis(w)
    k = k_lines.astype(np.float64) + CO.continuum(nu, w["T"], w["P"], x, table)
    edges = small_edges(nu)
    args = (k, w["depth_cm"], w["T"], w["t_surface"], nu, w["res"])
    for n_mu in (1, 2, 3, 4):
        mu, wt = quadrature(300 + L, n_mu)
        engine.set_flux_boundaries()
        engine.set_solar_source()
        check_fluxes(w, engine.atmosphere_fluxes(mu, wt, rows=True), FO.column_fluxes(*args, mu, wt))
        check_bands(engine.atmosphere_band_fluxes(mu, wt, edges), BO.band_fluxes(*args, mu, wt, edges),
                    band_floor(w, nu, edges))
        reflection = ("lambertian", "specular")[n_mu % 2]
        sun, mu_sun, t_top = SUNS["grid"], 0.5, 2.725
        engine.set_flux_boundaries(EPS_TABLES["table"], reflection, t_top)
        engine.set_solar_source(sun, mu_sun)
        ref = SO.solar_fluxes(*args, mu, wt, sun, mu_sun, EPS_TABLES["table"], reflection, t_top)
        check_solar(w, engine.atmosphere_fluxes(mu, wt, rows=True), ref, sun_floor(w, nu, sun, mu_sun))
        check_bands(engine.atmosphere_band_fluxes(mu, wt, edges),
                    SO.solar_band_fluxes(*args, mu, wt, edges, sun, mu_sun, EPS_TABLES["table"], reflection, t_top),
                    band_floor(w, nu, edges) + sun_floor(w, nu, sun, mu_sun, edges))


def everything(engine, mu, wt, edges):
    rad, tr = read_f32(engine)
    return [rad, tr, *engine.atmosphere_fluxes(mu, wt, rows=True), *engine.atmosphere_band_fluxes(mu, wt, edges)]


def assert_same_bits(a, b):
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


@pytest.mark.parametrize("L", [1, 8])
def test_no_continuum_and_a_cleared_one_give_the_plain_bits_and_launches(cengine, L):
    engine = cengine
    w = small_column(L)
    n = H.engine_setup(engine, w)
    mu, wt = quadrature(9, 3)
    edges = small_edges(axis(w))
    run_column(engine, w)
    never, launches = everything(engine, mu, wt, edges), engine.atmosphere_launches()
    k_never = kmatrix_f32(engine, L, n)
    engine.set_continuum(small_table(3), CO.synthetic_mole_fractions(3, L))
    run_column(engine, w)
    assert kmatrix_f32(engine, L, n).tobytes() != k_never.tobytes()
    engine.set_continuum()
    run_column(engine, w)
    assert_same_bits(everything(engine, mu, wt, edges), never)
    assert engine.atmosphere_launches() == launches
    assert kmatrix_f32(engine, L, n).tobytes() == k_never.tobytes()


@pytest.mark.parametrize("L", [1, 8])
@pytest.mark.parametrize("case", ["zero_table", "zero_x"])
def test_a_zero_continuum_changes_nothing(cengine, L, case):
    engine = cengine
    w = small_column(L)
    n = H.engine_setup(engine, w)
    mu, wt = quadrature(11, 2)
    edges = small_edges(axis(w))
    engine.set_flux_boundaries(EPS_TABLES["table"], "specular", 2.725)
    engine.set_solar_source(SUNS["part"], 0.5)
    run_column(engine, w)
    ref, k_ref = everything(engine, mu, wt, edges), kmatrix_f32(engine, L, n)
    table, x = small_table(5), CO.synthetic_mole_fractions(5, L)
    if case == "zero_table":
        table = dict(table, self=np.zeros_like(table["self"]), foreign=np.zeros_like(table["foreign"]))
    else:
        x = np.zeros(L)
    engine.set_continuum(table, x)
    run_column(engine, w)
    assert np.array_equal(kmatrix_f32(engine, L, n), k_ref)
    assert_same_bits(everything(engine, mu, wt, edges), ref)


def test_gas_cell_with_a_continuum_equals_the_separate_calls_and_the_oracle(cengine):
    """prb_gas_cell_host on a cell that takes the pipelined path without a continuum: with one, it takes
    upload_lines + set_grid + atmosphere(1 layer), bit for bit, and its spectra are the FP64 fold of k + k_c."""
    engine = cengine
    w = workloads.gas_cell(["h2o", "co2", "ch4", "o3"], 60000, 0.0, 1300.0, 0.001, 296, 1013.25,
                           [0.01, 400e-6, 1.8e-6, 5e-8], 10.0, 77)
    sp = w["species"]
    n = eng.grid_len(w["range_min"], w["range_max"], w["res"])
    assert n > 2 * 296 * 2048
    win = eng.window_len(w["cutoff"], w["res"])
    mol, q296, qt = [s.molmass for s in sp], [s.q296 for s in sp], [s.q(w["T"]) for s in sp]
    table = CO.synthetic_table(77, 0.0, 1300.0)
    x = [0.01]
    engine.upload_lines(w["lines"], n_groups=len(sp))
    engine.set_grid(w["range_min"], w["res"], n)
    engine.atmosphere([w["depth_cm"]], [w["T"]], [w["P"]], [w["conc"]], mol, [qt], q296, [win], 288.0, w["range_max"])
    k_lines = kmatrix_f32(engine, 1, n)
    engine.set_continuum(table, x)
    engine.atmosphere([w["depth_cm"]], [w["T"]], [w["P"]], [w["conc"]], mol, [qt], q296, [win], 288.0, w["range_max"])
    rad_ref, tr_ref = read_f32(engine)
    k_sep = kmatrix_f32(engine, 1, n)
    engine.gas_cell_host(w["lines"], len(sp), w["range_min"], w["res"], n, 0, n, w["depth_cm"], w["T"], w["P"], w["conc"],
                         mol, qt, q296, win, 288.0, w["range_max"])
    rad, tr = read_f32(engine)
    assert np.array_equal(rad, rad_ref, equal_nan=True) and np.array_equal(tr, tr_ref)
    assert np.array_equal(kmatrix_f32(engine, 1, n), k_sep)
    nu = ph.x_axis(w["range_min"], w["range_max"], w["res"])
    kc = CO.continuum(nu, [w["T"]], [w["P"]], x, table)
    check_kmatrix(k_sep, k_lines, kc)
    t = np.exp(-(k_sep[0].astype(np.float64)) * w["depth_cm"])
    I = ph.transmission(t, ph.planck_wavenumber(nu, 288.0), ph.planck_wavenumber(nu, w["T"]))
    ok = nu > 0
    np.testing.assert_allclose(rad[ok], I[ok], rtol=2e-5)
    assert np.abs(tr - t).max() <= H.T_ABS_TOL


def test_chunks_give_the_whole_grids_rows(cengine):
    engine = cengine
    w = small_column(24)
    table, x = small_table(13), CO.synthetic_mole_fractions(13, 24)
    n = H.engine_setup(engine, w)
    engine.set_continuum(table, x)
    run_column(engine, w)
    full = kmatrix_f32(engine, 24, n)
    rad_full, _ = read_f32(engine)
    parts, rads = [], []
    for a, b in ((0, 16384), (16384, n)):
        H.engine_setup(engine, w, a, b)
        run_column(engine, w)
        parts.append(kmatrix_f32(engine, 24, b - a))
        rads.append(read_f32(engine)[0])
    assert np.concatenate(parts, axis=1).tobytes() == full.tobytes()
    assert np.concatenate(rads).tobytes() == rad_full.tobytes()


def _set_raw(engine, table, x, n_table=None, t_ref=296.0, p_ref=1013.0, n_layers=None):
    dp = ctypes.POINTER(ctypes.c_double)
    arrs = [np.ascontiguousarray(table[k], dtype=np.float64) for k in ("nu", "self", "foreign", "texp")]
    x = np.ascontiguousarray(x, dtype=np.float64)
    return engine._lib.prb_set_continuum(engine._h, arrs[0].size if n_table is None else n_table,
                                         *[a.ctypes.data_as(dp) for a in arrs], t_ref, p_ref,
                                         x.size if n_layers is None else n_layers, x.ctypes.data_as(dp))


def test_argument_errors_keep_the_setting_and_layer_counts_must_match(cengine):
    engine = cengine
    w = small_column(3)
    n = H.engine_setup(engine, w)
    table, x = small_table(17), CO.synthetic_mole_fractions(17, 3)
    engine.set_continuum(table, x)
    run_column(engine, w)
    good = kmatrix_f32(engine, 3, n)
    nu = table["nu"]
    bad = [dict(n_table=1), dict(n_table=-1), dict(t_ref=0.0), dict(t_ref=np.nan), dict(p_ref=-1.0), dict(p_ref=np.inf),
           dict(n_layers=0)]
    for kw in bad:
        assert _set_raw(engine, table, x, **kw) == -2, kw                  # PRB_ERR_ARG
    broken = [dict(table, nu=nu[::-1].copy()), dict(table, nu=np.where(np.arange(nu.size) == 2, np.nan, nu)),
              dict(table, self=-table["self"]), dict(table, foreign=np.where(np.arange(nu.size) == 1, np.inf, table["foreign"])),
              dict(table, texp=np.where(np.arange(nu.size) == 0, np.nan, table["texp"]))]
    for t in broken:
        assert _set_raw(engine, t, x) == -2
    for xb in ([0.1, 1.5, 0.0], [0.1, -1e-9, 0.0], [np.nan, 0.1, 0.1]):
        assert _set_raw(engine, table, xb) == -2
    assert engine._lib.prb_set_continuum(engine._h, nu.size, None, None, None, None, 296.0, 1013.0, 3, None) == -2
    with pytest.raises(ValueError):
        engine.set_continuum(table, [0.5, 2.0, 0.0])
    run_column(engine, w)
    assert kmatrix_f32(engine, 3, n).tobytes() == good.tobytes()
    # a column of another layer count
    engine.set_continuum(table, [0.01, 0.02])
    with pytest.raises(_lib.EngineError, match="continuum") as ei:
        run_column(engine, w)
    assert ei.value.code == -2
    # n_table = 0 clears, NULL pointers allowed
    assert engine._lib.prb_set_continuum(engine._h, 0, None, None, None, None, 0.0, 0.0, 0, None) == 0
    run_column(engine, w)
    plain = kmatrix_f32(engine, 3, n)
    assert plain.tobytes() != good.tobytes()


def test_host_mirror_column_fluxes_with_a_continuum(data_root, engine, monkeypatch):
    """Atmosphere.columnFluxes(continuum=...) gives the bits of the engine-level call with the layers' H2O fractions
    (the same column replayed with set_continuum), the default is unchanged, and nothing leaks into the next call."""
    atm, rmin, rmax = _column_on_data_tree(data_root)
    mu, wt = FO.gauss_legendre_01(3)
    edges = np.linspace(rmin, rmax + 1.0, 5)
    table = CO.synthetic_table(29, rmin - 5.0, rmax + 5.0, spacing=2.0)
    calls = {}
    real_atm, real_range = engine.atmosphere, engine.set_layer_line_range
    monkeypatch.setattr(engine, "atmosphere", lambda *a: (calls.__setitem__("atm", a), real_atm(*a))[1])
    monkeypatch.setattr(engine, "set_layer_line_range",
                        lambda *a: (calls.__setitem__("range", a) if a else None, real_range(*a))[1])
    plain = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges)
    explicit = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges, continuum=None)
    wet = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges, continuum=table)
    h2o = [sum(m.concentration for m in l if not m.exotic and m.ID == 1) for l in atm]
    assert all(x > 0 for x in h2o)
    try:
        if "range" in calls:
            real_range(*calls["range"])
        engine.set_continuum(table, h2o)
        real_atm(*calls["atm"])
        up, down, ru, rd = engine.atmosphere_fluxes(mu, wt, rows=True)
        bu, bd = engine.atmosphere_band_fluxes(mu, wt, edges)
    finally:
        engine.set_continuum()
        real_range()
    for key, v in (("flux_up", up), ("flux_down", down), ("rad_up_top", ru), ("rad_down_surface", rd),
                   ("band_flux_up", bu), ("band_flux_down", bd)):
        np.testing.assert_array_equal(wet[key], v)
    after = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges)
    for key in plain:
        np.testing.assert_array_equal(explicit[key], plain[key])
        np.testing.assert_array_equal(after[key], plain[key])
    # this column is opaque next to the surface: the continuum shows above it
    assert not np.array_equal(wet["flux_up"], plain["flux_up"]) and not np.array_equal(wet["flux_down"], plain["flux_down"])
    rad_plain, _ = atm.columnSpectrum(288)
    rad_wet, _ = atm.columnSpectrum(288, continuum=table)
    assert not np.array_equal(rad_plain, rad_wet)
    with pytest.raises(ValueError, match="continuum"):
        atm.columnFluxes(288, continuum=dict(table, nu=table["nu"][::-1]))


def test_cfg4_full_size_continuum(cengine):
    """The 100-layer, 5 M-point cfg4 column with a synthetic table over 0-5000 cm-1 and its H2O profile: k-matrix points
    next to 0 cm-1, on both sides of block (1024-point), warp-span (128-point) and chunk edges, and at random, against
    the oracle on the same column's k matrix without the continuum; then the 3-node fluxes against an FP64 restatement
    run on the device over the device k matrix."""
    import torch
    engine = cengine
    w = workloads.atmosphere()
    n = H.engine_setup(engine, w)
    L = len(w["T"])
    assert n == 5_000_000 and L == 100
    table = CO.synthetic_table(4, 0.0, 5000.0)
    x = np.asarray(w["conc"])[:, 0]
    rng = np.random.default_rng(4)
    edges = [e + d for e in (128, 1024, 4096, 131072, 1 << 20, 2_500_000 - 2_500_000 % 1024) for d in (-2, -1, 0, 1)]
    idx = np.unique(np.concatenate([np.arange(0, 12), edges, rng.integers(0, n, 400), [n - 2, n - 1]]))
    idx_t = torch.as_tensor(idx, device="cuda")

    def sample():
        p, ld = engine.atmosphere_kmatrix_dev()
        return pd.device_tensor(p, L * ld).view(L, ld)[:, idx_t].cpu().numpy()

    engine.set_continuum()
    run_column(engine, w)
    k_lines = sample()
    mu, wt = FO.gauss_legendre_01(3)
    dry = engine.atmosphere_fluxes(mu, wt)
    engine.set_continuum(table, x)
    run_column(engine, w)
    k_dev = sample()
    nu_all = axis(w)
    kc = CO.continuum(nu_all[idx], w["T"], w["P"], x, table)
    check_kmatrix(k_dev, k_lines, kc)
    up, down = engine.atmosphere_fluxes(mu, wt)
    p, ld = engine.atmosphere_kmatrix_dev()
    kmat = pd.device_tensor(p, L * ld).view(L, ld)
    x0, dx, x_last, _ = eng.linspace_axis(w["range_min"], w["range_max"], n)
    h, c, kb = ph.h, ph.c, ph.k
    flt_max = float(np.finfo(np.float32).max)
    depth = [float(d) for d in w["depth_cm"]]
    r_up = torch.zeros(L + 1, dtype=torch.float64, device="cuda")
    r_down = torch.zeros(L + 1, dtype=torch.float64, device="cuda")
    floor = 0.0
    block = 1 << 20
    with torch.no_grad():
        for a in range(0, n, block):
            b = min(n, a + block)
            nu = torch.arange(a, b, dtype=torch.float64, device="cuda") * dx + x0
            if b == n:
                nu[-1] = x_last

            def planck(T):
                return 2E8 * h * c ** 2 * nu ** 3 / (torch.exp(100 * h * c * nu / kb / float(T)) - 1)

            B = [planck(T) for T in w["T"]]
            k = kmat[:, a:b].double()
            bs = planck(w["t_surface"])
            floor += float(ph.pi * torch.nan_to_num(bs).sum()) * w["res"]

            def add(r, j, f, I):
                r[j] += (torch.where(I.abs() <= flt_max, I, torch.zeros_like(I)) * f).sum()

            for m in range(3):
                f = 2 * ph.pi * wt[m] * mu[m] * w["res"]
                I = bs
                add(r_up, 0, f, I)
                for l in range(L):
                    t = torch.exp(-k[l] * depth[l] / mu[m])
                    I = t * I + (1 - t) * B[l]
                    add(r_up, l + 1, f, I)
                I = torch.zeros_like(nu)
                for l in range(L - 1, -1, -1):
                    t = torch.exp(-k[l] * depth[l] / mu[m])
                    I = t * I + (1 - t) * B[l]
                    add(r_down, l, f, I)
    floor *= 1e-7
    for got, ref in ((up, r_up.cpu().numpy()), (down, r_down.cpu().numpy())):
        err = np.abs(got - ref) / np.maximum(np.abs(ref), floor)
        assert err.max() <= 2e-5, (err.max(), int(err.argmax()))
    # the column is opaque next to the surface within FP32 (its surface fluxes do not move); the OLR does
    assert up[-1] != dry[0][-1]
