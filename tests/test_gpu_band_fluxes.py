"""GPU tests of the band fluxes (prb_atmosphere_band_fluxes -> k3_flux_tma's band pass / k3_flux_band_sum): per-band
level fluxes against the FP64 restatement (tests/band_flux_oracle.py) folded over the engine's own k matrix, the
one-band identity with prb_atmosphere_fluxes, partitions against the totals, repeatability, chunk invariance, independence
from other bands, argument errors, the host mirror (Atmosphere.columnFluxes(bands=...)) and the full-size cfg4 column."""
import numpy as np
import pytest

from oracle import physics as ph
from pyrad_b200 import _lib
from pyrad_b200 import classes as C
from pyrad_b200 import distributed as pd
from pyrad_b200 import engine as eng
from pyrad_b200 import workloads
from tests import band_flux_oracle as BO
from tests import flux_oracle as FO
from tests import helpers as H
from tests.test_gpu_fluxes import FLUX_FLOOR, FLUX_RTOL, data_root, device_kmatrix, quadrature, run_column, small_column  # noqa: F401

pytestmark = pytest.mark.gpu

#: RRTMG's 16 longwave bands, cm-1
RRTMG_LW = [10, 350, 500, 630, 700, 820, 980, 1080, 1180, 1390, 1480, 1800, 2080, 2250, 2380, 2600, 3250]


def axis(w):
    return ph.x_axis(w["range_min"], w["range_max"], w["res"])


def band_floor(w, nu, edges):
    """FLUX_FLOOR x pi sum_band B(nu, T_surface) res, per band."""
    idx = np.searchsorted(edges, nu, side="right") - 1
    sel = (idx >= 0) & (idx < len(edges) - 1)
    b = np.nan_to_num(ph.planck_wavenumber(nu, w["t_surface"]))
    return FLUX_FLOOR * ph.pi * np.bincount(idx[sel], weights=b[sel], minlength=len(edges) - 1) * w["res"]


def check_bands(got, ref, floor):
    for a, b in zip(got, ref):
        assert a.shape == b.shape
        err = np.abs(a - b)
        tol = FLUX_RTOL * np.abs(b) + floor[:, None]
        assert np.all(err <= tol), (np.argwhere(err > tol)[:5], (err / np.maximum(tol, 1e-300)).max())


def edge_sets(nu, seed):
    """The edge sets of the oracle comparison, on the axis nu of a small column (tens of thousands of points)."""
    step = nu[1] - nu[0]
    rng = np.random.default_rng(seed)
    n = nu.size
    return {
        "1_and_3_points": nu[[100, 101, 104, 127, 128, 131, 1023, 1024, 1027]],
        "127_128_129_points": nu[[256, 383, 511, 640, 768, 896]],
        "50_points": nu[300:n - 100:50][:200],
        "random": np.sort(rng.uniform(nu[0] - 1, nu[-1] + 1, 24)),
        "on_grid_values": nu[np.sort(rng.choice(n, 16, replace=False))],
        "outside_the_range": np.array([nu[0] - 100, nu[0] + 5.0, nu[-1] - 5.0, nu[-1] + 50, nu[-1] + 60]),
        "empty": np.array([nu[1000] + 0.1 * step, nu[1000] + 0.2 * step, nu[2000], nu[2000] + 0.5 * step,
                           nu[2000] + 0.7 * step, nu[3000]]),
        "whole": np.array([nu[0], nu[-1] + step]),
    }


@pytest.mark.parametrize("L", [1, 3, 8, 24])
def test_band_fluxes_match_the_fp64_fold_of_the_device_k_matrix(engine, L):
    w = small_column(L)
    n = H.engine_setup(engine, w)
    run_column(engine, w)
    k = device_kmatrix(engine, L, n)
    nu = axis(w)
    for n_mu in (1, 2, 3, 4):
        mu, wt = quadrature(200 + L, n_mu)
        for name, edges in edge_sets(nu, 10 * L + n_mu).items():
            got = engine.atmosphere_band_fluxes(mu, wt, edges)
            assert got[0].shape == got[1].shape == (len(edges) - 1, L + 1), name
            ref = BO.band_fluxes(k, w["depth_cm"], w["T"], w["t_surface"], nu, w["res"], mu, wt, edges)
            check_bands(got, ref, band_floor(w, nu, edges))
    empty = engine.atmosphere_band_fluxes(mu, wt, edge_sets(nu, 0)["empty"])
    assert np.all(empty[0][[0, 3]] == 0) and np.all(empty[1][[0, 3]] == 0) and np.all(empty[0][[1, 2, 4]] > 0)


def test_one_cm_bands_at_a_coarse_grid_where_every_span_crosses_an_edge(engine):
    w = workloads.atmosphere(n_layers=8, n_lines=6000, rmin=600.0, rmax=640.0, res=0.01, top_km=40.0)
    n = H.engine_setup(engine, w)
    run_column(engine, w)
    k = device_kmatrix(engine, 8, n)
    nu = axis(w)
    edges = np.arange(600.0, 642.0)                                 # 100-point bands; the last holds the point at 640
    mu, wt = FO.gauss_legendre_01(3)
    got = engine.atmosphere_band_fluxes(mu, wt, edges)
    check_bands(got, BO.band_fluxes(k, w["depth_cm"], w["T"], w["t_surface"], nu, w["res"], mu, wt, edges),
                band_floor(w, nu, edges))
    up, down = engine.atmosphere_fluxes(mu, wt)
    np.testing.assert_allclose(got[0].sum(axis=0), up, rtol=1e-6)
    np.testing.assert_allclose(got[1].sum(axis=0), down, rtol=1e-6)


@pytest.mark.parametrize("L", [1, 3, 24])
def test_one_band_over_the_whole_axis_is_the_total_flux(engine, L):
    """The FP32 stage is the same as prb_atmosphere_fluxes's; only the FP64 grouping of the sums differs."""
    w = small_column(L)
    H.engine_setup(engine, w)
    run_column(engine, w)
    for n_mu in (1, 2, 3, 4):
        mu, wt = quadrature(300 + L, n_mu)
        bu, bd = engine.atmosphere_band_fluxes(mu, wt, [w["range_min"], w["range_max"] + w["res"]])
        up, down = engine.atmosphere_fluxes(mu, wt)
        np.testing.assert_allclose(bu[0], up, rtol=1e-12, atol=0)
        np.testing.assert_allclose(bd[0], down, rtol=1e-12, atol=0)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_any_partition_adds_up_to_the_totals(engine, seed):
    w = small_column(24)
    H.engine_setup(engine, w)
    run_column(engine, w)
    rng = np.random.default_rng(seed)
    inner = np.sort(rng.uniform(w["range_min"], w["range_max"], [5, 60, 700][seed]))
    edges = np.concatenate([[w["range_min"]], inner, [w["range_max"] + w["res"]]])
    mu, wt = quadrature(seed, 3)
    bu, bd = engine.atmosphere_band_fluxes(mu, wt, edges)
    up, down = engine.atmosphere_fluxes(mu, wt)
    np.testing.assert_allclose(bu.sum(axis=0), up, rtol=1e-6)
    np.testing.assert_allclose(bd.sum(axis=0), down, rtol=1e-6)


def test_repeated_calls_give_identical_bits(engine):
    w = small_column(24)
    H.engine_setup(engine, w)
    run_column(engine, w)
    mu, wt = quadrature(3, 3)
    edges = np.sort(np.random.default_rng(4).uniform(w["range_min"], w["range_max"], 300))
    a = engine.atmosphere_band_fluxes(mu, wt, edges)
    b = engine.atmosphere_band_fluxes(mu, wt, edges)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


def test_chunks_give_their_bands_bit_for_bit(engine):
    """Two tile-aligned chunks on one engine (as test_chunks_add_up_to_the_whole_grid): a band inside a chunk gets the
    same bits from that chunk as from the whole grid; a band across the cut adds up to the whole grid's."""
    w = small_column(24)
    n = H.engine_setup(engine, w)
    nu = axis(w)
    step = nu[1] - nu[0]
    edges = np.array([nu[1000], nu[5000], nu[9000] + 0.5 * step, nu[15000], nu[18000], nu[20000], nu[30000]])
    inside0, across, inside1 = [0, 1, 2], [3], [4, 5]                # the cut is at point 16384
    mu, wt = quadrature(5, 3)
    run_column(engine, w)
    full = engine.atmosphere_band_fluxes(mu, wt, edges)
    parts = []
    for a, b in ((0, 16384), (16384, n)):
        H.engine_setup(engine, w, a, b)
        run_column(engine, w)
        parts.append(engine.atmosphere_band_fluxes(mu, wt, edges))
    for f in (0, 1):
        np.testing.assert_array_equal(parts[0][f][inside0], full[f][inside0])
        np.testing.assert_array_equal(parts[1][f][inside1], full[f][inside1])
        assert np.all(parts[1][f][inside0] == 0) and np.all(parts[0][f][inside1] == 0)
        np.testing.assert_allclose(parts[0][f][across] + parts[1][f][across], full[f][across], rtol=1e-12, atol=0)


def test_other_bands_leave_a_band_alone(engine):
    """A band on warp-span boundaries (multiples of 128 points) shares no span with its neighbours: its bits do not
    depend on which other bands are asked for, and asking for it alone reads only its own strips."""
    w = small_column(24)
    H.engine_setup(engine, w)
    run_column(engine, w)
    nu = axis(w)
    mu, wt = quadrature(6, 2)
    alone = engine.atmosphere_band_fluxes(mu, wt, nu[[4992, 6016]])
    many = engine.atmosphere_band_fluxes(mu, wt, nu[[100, 200, 4992, 6016, 30000, 30500]])
    dense = engine.atmosphere_band_fluxes(mu, wt, np.concatenate([nu[200:4993:7][:-1], nu[[4992, 6016]],
                                                                  nu[6016:39000:13][1:]]))
    i = int(np.flatnonzero(np.concatenate([nu[200:4993:7][:-1], nu[[4992, 6016]]]) == nu[4992])[0])
    for f in (0, 1):
        assert alone[f][0].tobytes() == many[f][2].tobytes() == dense[f][i].tobytes()


def test_argument_and_state_errors(engine):
    with eng.Engine(0) as fresh:
        with pytest.raises(_lib.EngineError) as ei:
            fresh.atmosphere_band_fluxes([1.0], [0.5], [600.0, 700.0])
        assert ei.value.code == -3                                  # PRB_ERR_STATE: no column yet
    w = small_column(3)
    H.engine_setup(engine, w)
    run_column(engine, w)
    good = [600.0, 620.0]
    bad = [([], [], good), ([0.5] * 5, [0.1] * 5, good), ([0.0], [0.5], good), ([1.5], [0.5], good),
           ([0.5], [-1.0], good), ([np.nan], [0.5], good), ([0.5], [0.5], []), ([0.5], [0.5], [600.0]),
           ([0.5], [0.5], [620.0, 600.0]), ([0.5], [0.5], [600.0, 600.0]), ([0.5], [0.5], [600.0, np.nan]),
           ([0.5], [0.5], [-np.inf, 600.0]), ([0.5], [0.5], [600.0, 610.0, np.inf])]
    for mu, wt, edges in bad:
        with pytest.raises(_lib.EngineError) as ei:
            engine.atmosphere_band_fluxes(mu, wt, edges)
        assert ei.value.code == -2, (mu, wt, edges)                 # PRB_ERR_ARG
    m, wq = np.array([0.5]), np.array([1.0])
    rc = engine._lib.prb_atmosphere_band_fluxes(engine._h, 1, m.ctypes.data_as(_lib.C.POINTER(_lib.C.c_double)),
                                                wq.ctypes.data_as(_lib.C.POINTER(_lib.C.c_double)), 1, None, None, None)
    assert rc == -2                                                 # NULL edges
    up, down = engine.atmosphere_band_fluxes([0.5], [1.0], good)    # and the engine still works
    assert up.shape == (1, 4) and np.all(np.isfinite(up)) and np.all(down[0, :-1] > 0) and down[0, -1] == 0


def test_host_mirror_band_fluxes(data_root):
    """Atmosphere.columnFluxes(bands=...) on a data tree: the totals are exactly those without bands, the bands add up
    to them, and band_heating_rate is heatingRate per band."""
    atm, rmin, rmax = _column_on_data_tree(data_root)
    mu, wt = FO.gauss_legendre_01(3)
    plain = atm.columnFluxes(288, mu=mu, weights=wt)
    edges = np.linspace(rmin, rmax + 1.0, 7)
    out = atm.columnFluxes(288, mu=mu, weights=wt, bands=edges)
    assert set(out) - set(plain) == {"band_edges", "band_flux_up", "band_flux_down", "band_net", "band_heating_rate"}
    for key, v in plain.items():
        np.testing.assert_array_equal(out[key], v)
    L = len(atm)
    assert out["band_flux_up"].shape == out["band_flux_down"].shape == (6, L + 1)
    assert out["band_heating_rate"].shape == (6, L)
    np.testing.assert_array_equal(out["band_edges"], edges)
    np.testing.assert_array_equal(out["band_net"], out["band_flux_up"] - out["band_flux_down"])
    np.testing.assert_allclose(out["band_flux_up"].sum(axis=0), out["flux_up"], rtol=1e-6)
    np.testing.assert_allclose(out["band_flux_down"].sum(axis=0), out["flux_down"], rtol=1e-6)
    for b in range(6):
        np.testing.assert_array_equal(out["band_heating_rate"][b], C.heatingRate(
            out["band_flux_up"][b], out["band_flux_down"][b], [l.depth for l in atm], [l.T for l in atm],
            [l.P for l in atm]))
    with pytest.raises(ValueError, match="bands"):
        atm.columnFluxes(288, bands=[rmax, rmin])


def _column_on_data_tree(root):
    """The 4-layer column of test_host_mirror_column_fluxes on the data tree at root."""
    from oracle import ref_harness as rh
    from pyrad_b200 import synth
    from tests import golden_util as G
    g = G.load("cell_fine_grid")
    species = [str(s) for s in g["species"]]
    for i, s in enumerate(species):
        sp = synth.species(s)
        ln = G.lines_of(g, i)
        rh.write_params(root, sp.global_iso, sp.name, sp.mol_id, 1, 0.99, sp.q296, 1, sp.molmass)
        rh.write_q_table(root, sp.global_iso, range(100, 501), [sp.q(t) for t in range(100, 501)])
        rh.write_line_segments(root, sp.global_iso, sp.mol_id, 1, ln, int(ln["nu"].min() / 100) * 100,
                               ln["nu"].max() + 101)
    C.BASE_RESOLUTION = float(g["base"])
    atm = C.Atmosphere("column")
    rmin, rmax = float(g["range_min"]), float(g["range_max"])
    for depth, T, P in ((2e4, 280, 800.0), (3e4, 250, 300.0), (5e4, 220, 40.0), (8e4, 230, 3.0)):
        layer = atm.addLayer(depth, T, P, rmin, rmax, dynamicResolution=False)
        for s, c in zip(species, g["conc"]):
            layer.addMolecule(s, concentration=float(c))
    return atm, rmin, rmax


def test_cfg4_full_size_band_fluxes(engine):
    """The 100-layer, 5 M-point cfg4 column with 3 Gauss-Legendre nodes, in RRTMG's 16 longwave bands and in 5000 bands
    of 1 cm-1 over 0-5000 cm-1, against the torch-FP64-on-device restatement of test_cfg4_full_size_fluxes_with_the_
    default_quadrature with per-band sums by index_add.  A band that holds a point where some layer has k < 0 (next to
    0 cm-1: the reference's negative Doppler widths) is held to the floor of the total-flux test instead of its own:
    there FP32 and FP64 transmittances above 1 part ways."""
    import torch
    w = workloads.atmosphere()
    n = H.engine_setup(engine, w)
    L = len(w["T"])
    assert n == 5_000_000 and L == 100
    run_column(engine, w)
    mu, wt = FO.gauss_legendre_01(3)
    sets = [np.array(RRTMG_LW, dtype=np.float64), np.arange(0.0, 5001.0)]
    got = [engine.atmosphere_band_fluxes(mu, wt, e) for e in sets]
    up, down = engine.atmosphere_fluxes(mu, wt)
    whole = engine.atmosphere_band_fluxes(mu, wt, [w["range_min"], w["range_max"] + w["res"]])
    np.testing.assert_allclose(whole[0][0], up, rtol=1e-12, atol=0)
    np.testing.assert_allclose(whole[1][0], down, rtol=1e-12, atol=0)
    p, ld = engine.atmosphere_kmatrix_dev()
    kmat = pd.device_tensor(p, L * ld).view(L, ld)
    x0, dx, x_last, _ = eng.linspace_axis(w["range_min"], w["range_max"], n)
    h, c, kb = ph.h, ph.c, ph.k
    flt_max = float(np.finfo(np.float32).max)
    depth = [float(d) for d in w["depth_cm"]]
    nb = [len(e) - 1 for e in sets]
    ref = [(torch.zeros(b + 1, L + 1, dtype=torch.float64, device="cuda"),
            torch.zeros(b + 1, L + 1, dtype=torch.float64, device="cuda")) for b in nb]
    pib = [torch.zeros(b + 1, dtype=torch.float64, device="cuda") for b in nb]
    kneg = [torch.zeros(b + 1, dtype=torch.bool, device="cuda") for b in nb]
    edges_t = [torch.as_tensor(e, device="cuda") for e in sets]
    block = 1 << 20
    with torch.no_grad():
        for a in range(0, n, block):
            b = min(n, a + block)
            nu = torch.arange(a, b, dtype=torch.float64, device="cuda") * dx + x0
            if b == n:
                nu[-1] = x_last

            def planck(T):
                return 2E8 * h * c ** 2 * nu ** 3 / (torch.exp(100 * h * c * nu / kb / float(T)) - 1)

            ids = []
            for s, et in enumerate(edges_t):
                i = torch.searchsorted(et, nu, right=True) - 1
                ids.append(torch.where((i >= 0) & (i < nb[s]), i, torch.full_like(i, nb[s])))   # nb[s]: no band
            B = [planck(T) for T in w["T"]]
            k = kmat[:, a:b].double()
            neg = (k < 0).any(dim=0)
            bs = torch.nan_to_num(planck(w["t_surface"]))
            for s in range(2):
                pib[s].index_add_(0, ids[s], bs)
                kneg[s][ids[s][neg]] = True

            def level_add(r, j, f, I):
                I = torch.where(I.abs() <= flt_max, I, torch.zeros_like(I)) * f
                for s in range(2):
                    r[s][:, j].index_add_(0, ids[s], I)

            for i in range(3):
                f = 2 * ph.pi * wt[i] * mu[i] * w["res"]
                I = planck(w["t_surface"])
                level_add([r[0] for r in ref], 0, f, I)
                for l in range(L):
                    t = torch.exp(-k[l] * depth[l] / mu[i])
                    I = t * I + (1 - t) * B[l]
                    level_add([r[0] for r in ref], l + 1, f, I)
                I = torch.zeros_like(nu)
                for l in range(L - 1, -1, -1):
                    t = torch.exp(-k[l] * depth[l] / mu[i])
                    I = t * I + (1 - t) * B[l]
                    level_add([r[1] for r in ref], l, f, I)
    total_floor = FLUX_FLOOR * ph.integrate_spectrum(
        ph.planck_wavenumber(ph.x_axis(w["range_min"], w["range_max"], w["res"]), w["t_surface"]), ph.pi, w["res"])
    for s in range(2):
        floor = FLUX_FLOOR * ph.pi * pib[s][:-1].cpu().numpy() * w["res"]
        floor = np.where(kneg[s][:-1].cpu().numpy(), total_floor, floor)
        check_bands(got[s], [r[:-1].cpu().numpy() for r in ref[s]], floor)
    assert np.all(got[0][1][:, -1] == 0) and np.all(got[1][1][:, -1] == 0)    # nothing comes down at the top
    np.testing.assert_allclose(got[0][0].sum(axis=0), got[1][0][10:3250].sum(axis=0), rtol=1e-6)
