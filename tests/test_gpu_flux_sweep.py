"""Seeded random sweep of the column flux path (prb_atmosphere, then prb_atmosphere_fluxes / prb_atmosphere_band_fluxes
with or without boundaries, a Sun and a continuum) against the FP64 restatements, and the rule that a grid change drops
the resident column.

Each case draws a grid (0 cm-1 to 5000 cm-1, 0.001 to 0.1 cm-1, 1 to ~300k points), a chunk of it (the whole grid, or an
unaligned slice down to 0 points), 1 to 40 layers with either layer fold, a temperature profile (noisy standard, random,
isothermal: inversions and layers warmer than the surface), a depth scale from transparent to opaque, a quadrature of 1
to 4 nodes, and the flux options, all together: so that the Planck paths of k3_flux_tma (interpolated, per point, the
expm1 branch, the grids where the host never interpolates), its strip and row-group walks and the chunk edges meet in
combinations the fixed tests do not list.  The device k matrix is held fixed (it is the line sum's, compared elsewhere:
test_gpu_fuzz.py) and everything after it is compared with tests/solar_flux_oracle.py over the chunk's own axis.
PRB_FUZZ_SCALE scales the case counts as in test_gpu_fuzz.py."""
import os

import numpy as np
import pytest

from oracle import physics as ph
from pyrad_b200 import _lib
from pyrad_b200 import engine as eng
from pyrad_b200 import workloads
from tests import continuum_oracle as CO
from tests import flux_oracle as FO
from tests import helpers as H
from tests import solar_flux_oracle as SO
from tests.test_gpu_band_fluxes import band_floor, check_bands
from tests.test_gpu_fluxes import FLUX_FLOOR, FLUX_RTOL, ROWS_RTOL, device_kmatrix, run_column, small_column
from tests.test_gpu_solar_flux import sun_floor

SCALE = int(os.environ.get("PRB_FUZZ_SCALE", "1"))
RMINS = (0.0, 0.5, 20.0, 600.0, 2300.0, 4000.0)
RESES = (0.001, 0.002, 0.005, 0.01, 0.05, 0.1)
CHUNK_LENGTHS = (0, 1, 3, 4, 5, 1023, 1024, 1025)
NU_MAX = 5000.0             # with T >= 150 K every B and row stays far above FP32's flush-to-zero range
T_MIN, T_MAX = 150.0, 340.0
SPLIT = 16384               # chunk edges at which the k matrix is shard invariant (test_chunks_add_up_to_the_whole_grid)
K3T_MINB = 5                # k3_fold_tma's resident CTAs per SM (csrc/k3_stream.cuh): the fold loops over strips beyond
K3T_STRIP = 1024            # K3T_MINB x SMs strips of K3T_STRIP points
N_CASES = 48


# ---------------------------------------------------------------------------------------------------- drawing cases
def draw_params(seed, n_max=300_000, n_min=1, L=None, whole=False):
    """The parameters of case `seed` (no workload yet: cheap, so that the sweep's coverage is checked on the CPU)."""
    rng = np.random.default_rng(9100 + seed)
    rmin = float(rng.choice(RMINS))
    res = float(rng.choice([r for r in RESES if rmin + (n_min + 2) * r <= NU_MAX]))
    n = int(np.exp(rng.uniform(np.log(n_min), np.log(max(n_max, n_min + 1)))))
    n = max(n_min, min(n, int((NU_MAX - rmin) / res) - 2))
    rmax = rmin + (n + 0.5) * res                                   # int((rmax - rmin) / res) == n
    assert eng.grid_len(rmin, rmax, res) == n
    # chunk: the whole grid, or [a, b) of a listed or random length, mostly starting off a multiple of 4
    a, b = 0, n
    if not whole and rng.random() < 0.7:
        m = CHUNK_LENGTHS[seed % len(CHUNK_LENGTHS)] if rng.random() < 0.6 else int(rng.integers(0, n + 1))
        m = min(m, n)
        a = int(rng.integers(0, n - m + 1))
        if a % 4 == 0 and a + m < n and rng.random() < 0.8:
            a += int(rng.integers(1, min(3, n - m - a) + 1))
        b = a + m
    L = int(rng.integers(1, 41)) if L is None else L
    t_mode = ("profile", "random", "isothermal")[seed % 3]
    p = dict(seed=seed, rmin=rmin, res=res, rmax=rmax, n=n, chunk=(a, b), L=L, tma=int(rng.random() < 0.7),
             t_mode=t_mode, t_noise=rng.normal(0.0, 10.0, L), t_random=rng.uniform(T_MIN, T_MAX, L),
             t_iso=float(rng.uniform(T_MIN, T_MAX)), t_surface=float(rng.uniform(200.0, 330.0)),
             depth_scale=float(np.exp(rng.uniform(np.log(1e-7), np.log(1e-2)))), top_km=float(rng.uniform(10.0, 80.0)))
    n_mu = int(rng.integers(1, 5))
    mu = 1.0 - rng.uniform(0.0, 0.98, n_mu)                        # (0.02, 1]
    if rng.random() < 0.3:
        mu[int(rng.integers(0, n_mu))] = 1.0
    p.update(mu=mu, wt=rng.uniform(0.05, 0.5, n_mu))
    # options, drawn independently; tables over the grid's span (and beyond it)
    x0, x1 = rmin, rmax
    span = max(x1 - x0, 1.0)
    kind = str(rng.choice(["none", "constant", "table"]))
    eps = None
    if kind == "constant":
        eps = float(rng.choice([0.0, rng.uniform(0, 1), 1.0]))
    elif kind == "table":
        m = int(rng.integers(2, 8))
        tn = np.sort(rng.uniform(x0 - 0.2 * span, x1 + 0.2 * span, m))
        te = rng.uniform(0.0, 1.0, m)
        te[rng.random(m) < 0.15] = 0.0
        te[rng.random(m) < 0.15] = 1.0
        eps = (tn, te)
    p.update(eps=eps, reflection=str(rng.choice(["lambertian", "specular"])),
             t_top=float(rng.choice([0.0, 2.725, 250.0])))
    sun_kind = str(rng.choice(["none", "partial", "full"]))
    sun, mu_sun = None, 1.0
    if sun_kind != "none":
        m = int(rng.integers(2, 7))
        if sun_kind == "full":
            lo, hi = x0 - 0.3 * span - 1.0, x1 + 0.3 * span + 1.0
        else:                                    # over the middle of the grid only
            lo = x0 + 0.2 * (x1 - x0)
            hi = max(x0 + 0.7 * (x1 - x0), lo + 0.5 * res)
        tn = np.sort(rng.uniform(lo, hi, m))
        tn[0], tn[-1] = lo, hi
        tn = np.unique(tn)
        scale = ph.pi * float(ph.planck_wavenumber(max(0.5 * (x0 + x1), 1.0), p["t_surface"]))
        sun = (tn, scale * rng.uniform(0.0, 3.0, tn.size))
        mu_sun = float(1.0 - rng.uniform(0.0, 0.98))
    p.update(sun_kind=sun_kind, sun=sun, mu_sun=mu_sun, continuum=bool(rng.random() < 0.3),
             bands=bool(rng.random() < 0.6), band_seed=int(rng.integers(0, 2 ** 31)))
    return p


def band_edges(p, nu_all):
    """Random edges on the grid's axis: grid values around the chunk, a single-point band, an empty band (two edges
    between neighbouring points) and edges outside the grid."""
    rng = np.random.default_rng(p["band_seed"])
    n = nu_all.size
    a, b = p["chunk"]
    step = nu_all[1] - nu_all[0] if n > 1 else p["res"]
    idx = rng.integers(max(a - 2, 0), min(b + 2, n), 6) if b > a else rng.integers(0, n, 6)
    e = list(nu_all[idx])
    i = int(idx[0])
    if i + 1 < n:
        e += [nu_all[i], nu_all[i + 1]]                              # a band of exactly one point
        j = int(idx[1]) if int(idx[1]) + 1 < n else i
        e += [nu_all[j] + 0.25 * (nu_all[j + 1] - nu_all[j]), nu_all[j] + 0.6 * (nu_all[j + 1] - nu_all[j])]   # empty
    e += [nu_all[0] - rng.uniform(0.1, 50.0) * step, nu_all[-1] + rng.uniform(0.1, 50.0) * step]
    e += list(rng.uniform(nu_all[0] - step, nu_all[-1] + step, int(rng.integers(0, 4))))
    return np.unique(np.asarray(e, dtype=np.float64))


def build_column(p):
    """The workload of a case: the standard column of p['L'] layers on the case's grid, its T and depth replaced.  One
    line per 0.25 cm-1 keeps k > 0 at every point of the bottom layers (no point of the column is left transparent)."""
    n_lines = int(min(max(4 * (p["rmax"] - p["rmin"] + 10.0), 40), 40000))
    w = workloads.atmosphere(n_layers=p["L"], n_lines=n_lines, rmin=p["rmin"], rmax=p["rmax"], res=p["res"],
                             top_km=p["top_km"], seed=4000 + p["seed"])
    if p["t_mode"] == "profile":
        w["T"] = np.clip(w["T"] + p["t_noise"], T_MIN, T_MAX)
    elif p["t_mode"] == "random":
        w["T"] = p["t_random"].copy()
    else:
        w["T"] = np.full(p["L"], p["t_iso"])
    w["t_surface"] = p["t_surface"]
    w["depth_cm"] = w["depth_cm"] * p["depth_scale"]
    return w


def describe(p):
    keep = ("seed", "rmin", "res", "n", "chunk", "L", "tma", "t_mode", "t_surface", "depth_scale", "mu", "wt", "eps",
            "reflection", "t_top", "sun_kind", "mu_sun", "continuum", "bands")
    return {k: p[k] for k in keep}


# ---------------------------------------------------------------------------------------------------- running a case
def run_case(engine, p, w, chunk=None):
    """Upload, set the grid and run the column (the continuum, when drawn, only for this call)."""
    a, b = p["chunk"] if chunk is None else chunk
    engine.upload_lines(w["lines"], n_groups=len(w["species"]))
    engine.set_grid(p["rmin"], p["res"], p["n"], a, b)
    engine.set_option(eng.OPT_FOLD_TMA, p["tma"])
    if p["continuum"]:
        engine.set_continuum(CO.synthetic_table(p["seed"], p["rmin"] - 1.0, p["rmax"] + 1.0,
                                                spacing=max((p["rmax"] - p["rmin"]) / 6, 0.05)),
                             CO.synthetic_mole_fractions(p["seed"], p["L"]))
    try:
        run_column(engine, w)
    finally:
        engine.set_option(eng.OPT_FOLD_TMA, 1)
        engine.set_continuum()


def set_options(engine, p):
    engine.set_flux_boundaries(p["eps"], p["reflection"], p["t_top"])
    engine.set_solar_source(p["sun"], p["mu_sun"])


def clear_options(engine):
    engine.set_solar_source()
    engine.set_flux_boundaries()


def thermal_floor(w, nu):
    """FLUX_FLOOR x pi sum B(nu, T_surface) res over the chunk's axis (check_solar's floor, per chunk)."""
    return FLUX_FLOOR * ph.pi * float(np.sum(np.nan_to_num(ph.planck_wavenumber(nu, w["t_surface"])))) * w["res"]


def oracle_row_bound(nu, T, t_surface, t_top, sun, L):
    """An upper bound of the FP64 oracle's own absolute error in a row, per point.  Layer.transmission forms the emission
    weight as 1 - exp(-tau): exp is good to 2^-52 and the subtraction is exact, so the weight is off by up to 2^-52 in
    ABSOLUTE terms -- all of it when tau < ~1e-12 (a nearly transparent layer), where the device's thin-layer series is
    the accurate side.  Each layer adds at most 2 x 2^-52 of the largest source (emission weight and transmitted part),
    over both passes and the reflection: (4 L + 4) 2^-52 max(B(T_l), B(T_s), B(T_top), S).  Rows that such a layer does
    not dominate are 1e8 and more above it, so the bound changes nothing else."""
    with np.errstate(all="ignore"):
        src = [ph.planck_wavenumber(nu, t) for t in (*T, t_surface)]
        if t_top > 0:
            src.append(ph.planck_wavenumber(nu, t_top))
    src.append(SO.irradiance(nu, sun))
    return (4 * L + 4) * 2.0 ** -52 * np.nanmax(np.array(src), axis=0)


def assert_rows(got, ref, bound, info):
    err = np.abs(got - ref)
    tol = ROWS_RTOL * np.abs(ref) + bound
    assert np.all(err <= tol), (info, int(np.sum(err > tol)), float(np.max((err - bound) / np.abs(ref))))


def check_case(engine, p, w):
    """Run case p on the engine and compare everything after the k matrix with the FP64 restatements."""
    info = describe(p)
    a, b = p["chunk"]
    nc, L = b - a, p["L"]
    nu_all = ph.x_axis(p["rmin"], p["rmax"], p["res"])
    assert nu_all.size == p["n"]
    nu = nu_all[a:b]
    mu, wt = p["mu"], p["wt"]
    edges = band_edges(p, nu_all) if p["bands"] else None
    run_case(engine, p, w)
    if nc == 0:                                  # an empty chunk contributes nothing, whatever is set
        rad, tr = engine.atmosphere_read()
        assert rad.shape == tr.shape == (0,), info
        set_options(engine, p)
        try:
            up, down, ru, rd = engine.atmosphere_fluxes(mu, wt, rows=True)
            assert ru.shape == rd.shape == (mu.size, 0) and not up.any() and not down.any(), info
            if edges is not None:
                bu, bd = engine.atmosphere_band_fluxes(mu, wt, edges)
                assert bu.shape == (edges.size - 1, L + 1) and not bu.any() and not bd.any(), info
        finally:
            clear_options(engine)
        return
    k = device_kmatrix(engine, L, nc)
    depth, T, ts = w["depth_cm"], w["T"], w["t_surface"]
    ok = (nu > 0) & np.all(k >= 0, axis=0)       # rows: away from 0 cm-1 and the points next to it where k < 0
    # prb_atmosphere's own radiance and transmittance: the oracle's fold at mu = 1
    rad, tr = engine.atmosphere_read()
    _, _, r_rad, _ = FO.column_fluxes(k, depth, T, ts, nu, w["res"], [1.0], [0.5])
    bound = oracle_row_bound(nu, T, ts, p["t_top"], p["sun"], L)[ok]
    assert_rows(rad[ok], r_rad[0][ok], bound, info)
    t_ref = np.prod(np.exp(-k * np.asarray(depth)[:, None]), axis=0)
    dt = np.abs(tr[ok] - t_ref[ok])
    assert dt.size == 0 or dt.max() <= H.T_ABS_TOL, (info, float(dt.max()))
    # the vertical node without boundaries or Sun is the column's radiance, bit for bit
    _, _, ru1, _ = engine.atmosphere_fluxes([1.0], [0.5], rows=True)
    rad32 = np.empty(nc, dtype=np.float32)
    engine.atmosphere_read_f32(rad32, None)
    np.testing.assert_array_equal(ru1[0], rad32, err_msg=str(info))
    # the drawn quadrature and options
    set_options(engine, p)
    try:
        up, down, ru, rd = engine.atmosphere_fluxes(mu, wt, rows=True)
        bands = engine.atmosphere_band_fluxes(mu, wt, edges) if edges is not None else None
    finally:
        clear_options(engine)
    args = (k, depth, T, ts, nu, w["res"], mu, wt)
    opts = dict(sun=p["sun"], mu_sun=p["mu_sun"], eps_table=p["eps"], reflection=p["reflection"], t_top=p["t_top"])
    r_up, r_down, r_ru, r_rd = SO.solar_fluxes(*args, **opts)
    assert_rows(ru[:, ok], r_ru[:, ok], bound, info)
    assert_rows(rd[:, ok], r_rd[:, ok], bound, info)
    floor = thermal_floor(w, nu) + sun_floor(w, nu, p["sun"], p["mu_sun"])
    for name, x, y in (("up", up, r_up), ("down", down, r_down)):
        err = np.abs(x - y)
        assert np.all(err <= FLUX_RTOL * np.abs(y) + floor), (info, name, float((err / np.maximum(np.abs(y), floor)).max()))
    if edges is not None:
        ref = SO.solar_band_fluxes(*args[:6], mu, wt, edges, **opts)
        try:
            check_bands(bands, ref, band_floor(w, nu, edges) + sun_floor(w, nu, p["sun"], p["mu_sun"], edges))
        except AssertionError as ex:
            raise AssertionError((info, list(edges), str(ex))) from None


# ---------------------------------------------------------------------------------------------------- the sweep
def test_the_sweep_draws_every_path():
    """The cases at scale 1 meet every grid, chunk, layer and option class the sweep is for (CPU only: no workload)."""
    ps = [draw_params(s) for s in range(N_CASES)]
    assert {p["rmin"] for p in ps} == set(RMINS) and {p["res"] for p in ps} == set(RESES)
    lengths = {p["chunk"][1] - p["chunk"][0] for p in ps if p["chunk"] != (0, p["n"])}
    assert set(CHUNK_LENGTHS) <= lengths
    assert any(p["chunk"][0] % 4 for p in ps) and any(p["chunk"] == (0, p["n"]) for p in ps)
    assert {p["L"] % 4 for p in ps if p["tma"] and p["L"] >= 4} == {0, 1, 2, 3}
    assert {p["L"] for p in ps if p["L"] <= 3} == {1, 2, 3} and {p["tma"] for p in ps} == {0, 1}
    assert {p["mu"].size for p in ps} == {1, 2, 3, 4} and any(1.0 in p["mu"] for p in ps)
    assert {p["t_mode"] for p in ps} == {"profile", "random", "isothermal"}
    rnd = [p for p in ps if p["t_mode"] == "random" and p["L"] > 1]
    assert any(np.any(np.diff(p["t_random"]) > 0) for p in rnd)                     # inversions
    assert any(np.any(p["t_random"] > p["t_surface"]) for p in rnd)                 # layers warmer than the surface
    assert {type(p["eps"]).__name__ for p in ps} == {"NoneType", "float", "tuple"}
    assert {p["reflection"] for p in ps} == {"lambertian", "specular"} and {p["t_top"] for p in ps} == {0.0, 2.725, 250.0}
    assert {p["sun_kind"] for p in ps} == {"none", "partial", "full"}
    assert any(p["continuum"] for p in ps) and any(p["bands"] for p in ps)
    assert any(p["n"] == 1 for p in ps) and max(p["n"] for p in ps) > 50_000
    # the host's interpolation rule (prb_atmosphere): never on coarse grids, switched on inside a grid from 0 cm-1
    c2 = CO.C2
    coarse = [p for p in ps if p["tma"] and p["L"] >= 4 and (3 * p["res"]) ** 2 / 8 * (c2 / T_MIN) ** 2 > 1e-7]
    assert coarse and any(p["rmin"] < 1 for p in ps if p["n"] > 1 and p["chunk"][0] == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(N_CASES * SCALE))
def test_random_column_fluxes_match_the_oracle(engine, seed):
    p = draw_params(seed)
    check_case(engine, p, build_column(p))


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3 + SCALE // 5))
def test_columns_that_loop_over_strips(engine, seed):
    """More than K3T_MINB x SMs strips: the fold's CTAs and both flux grids loop over strips, with one row group per strip
    (L <= 4) or a ragged last group (L mod 4 != 0)."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n_min = K3T_MINB * sms * K3T_STRIP + 1
    p = draw_params(50_000 + seed, n_max=int(1.2 * n_min), n_min=n_min, L=(4, 9, 1, 6, 3, 7)[seed % 6], whole=True)
    p["tma"] = 1
    assert p["n"] >= n_min and (p["n"] + K3T_STRIP - 1) // K3T_STRIP > K3T_MINB * sms
    check_case(engine, p, build_column(p))


@pytest.mark.gpu
@pytest.mark.parametrize("rmin,res,L,tma", [(600.0, 0.1, 1, 1), (0.5, 0.05, 3, 1), (2300.0, 0.01, 8, 1),
                                            (4000.0, 0.002, 5, 0)])
def test_a_one_point_grid(engine, rmin, res, L, tma):
    """np.linspace(range_min, range_max, 1) is [range_min]: the one point's Planck term is taken there, not at
    range_max (found by the sweep: the fold and the flux passes took the axis' last value, range_max)."""
    p = draw_params(70_000 + L, whole=True)
    p.update(rmin=rmin, res=res, rmax=rmin + 1.5 * res, n=1, chunk=(0, 1), L=L, tma=tma, t_mode="random",
             t_random=np.linspace(T_MIN, T_MAX, L), t_noise=np.zeros(L), bands=True, continuum=False)
    check_case(engine, p, build_column(p))


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(4 * SCALE))
def test_aligned_chunks_add_up_to_the_whole_grid(engine, seed):
    """2 or 3 chunks cut at multiples of SPLIT, a Sun and boundaries set: the rows concatenate bit for bit, and the
    totals and bands of the chunks add up to the whole grid's (only the FP64 grouping of the sums differs)."""
    p = draw_params(80_000 + seed, n_max=6 * SPLIT, n_min=2 * SPLIT + 1, whole=True)
    p["continuum"] = bool(seed % 2)
    if p["sun"] is None:
        p["sun"], p["mu_sun"] = ([p["rmin"] - 1.0, p["rmax"] + 1.0], [0.3, 0.6]), 0.5
    if p["eps"] is None:
        p["eps"] = 0.7
    rng = np.random.default_rng(seed)
    cuts = sorted(rng.choice(np.arange(1, (p["n"] - 1) // SPLIT + 1), size=int(rng.integers(1, 3)), replace=False))
    bounds = [0] + [int(c) * SPLIT for c in np.unique(cuts)] + [p["n"]]
    w = build_column(p)
    nu_all = ph.x_axis(p["rmin"], p["rmax"], p["res"])
    edges = band_edges(p, nu_all)
    mu, wt = p["mu"], p["wt"]

    def everything(chunk):
        run_case(engine, p, w, chunk)
        set_options(engine, p)
        try:
            return engine.atmosphere_fluxes(mu, wt, rows=True), engine.atmosphere_band_fluxes(mu, wt, edges)
        finally:
            clear_options(engine)

    full, full_b = everything((0, p["n"]))
    parts = [everything((a, b)) for a, b in zip(bounds[:-1], bounds[1:])]
    info = (describe(p), bounds)
    for r in (2, 3):
        np.testing.assert_array_equal(np.concatenate([x[0][r] for x in parts], axis=1), full[r], err_msg=str(info))
    for f in (0, 1):
        np.testing.assert_allclose(sum(x[0][f] for x in parts), full[f], rtol=1e-12, atol=0, err_msg=str(info))
        np.testing.assert_allclose(sum(x[1][f] for x in parts), full_b[f], rtol=1e-12, atol=0, err_msg=str(info))


# ---------------------------------------------------------------------------------------------------- the resident column
def _readers(e):
    n = e.n_chunk
    return {
        "read": lambda: e.atmosphere_read(),
        "read_f32": lambda: e.atmosphere_read_f32(np.empty(n, dtype=np.float32), np.empty(n, dtype=np.float32)),
        "result_dev": lambda: e.atmosphere_result_dev(),
        "kmatrix_dev": lambda: e.atmosphere_kmatrix_dev(),
        "integrate": lambda: e.atmosphere_integrate(np.pi, 0.001),
        "fluxes": lambda: e.atmosphere_fluxes([0.5], [1.0], rows=True),
        "band_fluxes": lambda: e.atmosphere_band_fluxes([0.5], [1.0], [600.0, 620.0, 640.0]),
    }


def assert_no_column(e, why):
    for name, fn in _readers(e).items():
        with pytest.raises(_lib.EngineError) as ei:
            fn()
        assert ei.value.code == -3, (why, name)                     # PRB_ERR_STATE


STATE_SUN = ([590.0, 615.0, 650.0], [0.2, 0.6, 0.3])
STATE_EPS = ([600.0, 620.0, 640.0], [0.9, 0.4, 0.8])


def _state_settings(e, L):
    e.set_flux_boundaries(STATE_EPS, "specular", 2.725)
    e.set_solar_source(STATE_SUN, 0.6)
    e.set_continuum(CO.synthetic_table(5, 590.0, 650.0), CO.synthetic_mole_fractions(5, L))


def _column_results(e, L):
    mu, wt = FO.gauss_legendre_01(2)
    rad, tr = e.atmosphere_read()
    k = device_kmatrix(e, L, e.n_chunk)
    return [rad, tr, k, *e.atmosphere_fluxes(mu, wt, rows=True), *e.atmosphere_band_fluxes(mu, wt, [600.0, 611.0, 640.0])]


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", ["same", "shorter", "longer"])
def test_a_grid_change_drops_the_resident_column(engine, chunk):
    """After prb_set_grid every column reader refuses (PRB_ERR_STATE) until prb_atmosphere runs again; then the readers
    give a fresh engine's bits, and the boundaries, the Sun and the continuum set before the grid change still apply."""
    w = small_column(3)
    n = eng.grid_len(w["range_min"], w["range_max"], w["res"])
    first = (0, 24576)
    second = {"same": first, "shorter": (4096, 12288), "longer": (0, n)}[chunk]
    try:
        H.engine_setup(engine, w, *first)
        _state_settings(engine, 3)
        run_column(engine, w)
        _column_results(engine, 3)                                  # readable
        engine.set_grid(w["range_min"], w["res"], n, *second)
        assert_no_column(engine, ("after set_grid", chunk))
        run_column(engine, w)
        got = _column_results(engine, 3)
        with eng.Engine(0) as fresh:
            H.engine_setup(fresh, w, *second)
            _state_settings(fresh, 3)
            run_column(fresh, w)
            want = _column_results(fresh, 3)
            fresh.set_solar_source()
            fresh.set_flux_boundaries()
            fresh.set_continuum()
            run_column(fresh, w)
            plain = _column_results(fresh, 3)
    finally:
        engine.set_continuum()
        clear_options(engine)
    for i, (x, y) in enumerate(zip(got, want)):
        assert x.tobytes() == y.tobytes(), (chunk, i)
    # (the settings matter: the continuum changes k, the Sun flux_down, the boundaries the upward rows)
    assert got[2].tobytes() != plain[2].tobytes() and got[4][-1] != plain[4][-1] and got[5].tobytes() != plain[5].tobytes()


@pytest.mark.gpu
def test_gas_cell_host_leaves_a_readable_column(engine):
    """prb_gas_cell_host sets the grid itself and leaves the column of the separate calls, readable."""
    w = workloads.gas_cell(["co2", "h2o"], 4000, 600.0, 640.0, 0.001, 260, 800.0, [400e-6, 0.01], 10.0, 31)
    sp = w["species"]
    n = eng.grid_len(w["range_min"], w["range_max"], w["res"])
    mol, q296, qt = [s.molmass for s in sp], [s.q296 for s in sp], [s.q(w["T"]) for s in sp]
    win = eng.window_len(w["cutoff"], w["res"])
    engine.upload_lines(w["lines"], n_groups=len(sp))
    engine.set_grid(w["range_min"], w["res"], n, 1000, 9000)
    assert_no_column(engine, "before gas_cell_host")
    engine.gas_cell_host(w["lines"], len(sp), w["range_min"], w["res"], n, 3, n - 5, w["depth_cm"], w["T"], w["P"],
                         w["conc"], mol, qt, q296, win, 288.0, w["range_max"])
    got = [*engine.atmosphere_read(), *engine.atmosphere_fluxes([1.0], [0.5])]
    engine.set_grid(w["range_min"], w["res"], n, 3, n - 5)
    engine.atmosphere([w["depth_cm"]], [w["T"]], [w["P"]], [w["conc"]], mol, [qt], q296, [win], 288.0, w["range_max"])
    want = [*engine.atmosphere_read(), *engine.atmosphere_fluxes([1.0], [0.5])]
    assert got[0].size == n - 8
    for i, (x, y) in enumerate(zip(got, want)):
        assert x.tobytes() == y.tobytes(), i


@pytest.mark.gpu
def test_a_failed_atmosphere_leaves_no_column(engine):
    w = small_column(3)
    H.engine_setup(engine, w)
    run_column(engine, w)
    good = engine.atmosphere_read()
    sp = w["species"]
    qt = np.array([[s.q(T) for s in sp] for T in w["T"]])
    with pytest.raises(_lib.EngineError) as ei:                     # a window of no points fails the argument check
        engine.atmosphere(w["depth_cm"], w["T"], w["P"], w["conc"], [s.molmass for s in sp], qt, [s.q296 for s in sp],
                          [0, 0, 0], w["t_surface"], w["range_max"])
    assert ei.value.code == -2
    assert_no_column(engine, "after a failed atmosphere")
    run_column(engine, w)
    again = engine.atmosphere_read()
    assert good[0].tobytes() == again[0].tobytes() and good[1].tobytes() == again[1].tobytes()
