"""GPU tests of the column fluxes (prb_atmosphere_fluxes -> k3_flux_tma / k3_flux_sum): level fluxes and slant radiances
against the FP64 restatement (tests/flux_oracle.py) folded over the engine's own k matrix and over the oracle's k, the
bitwise identity with prb_atmosphere's radiance at mu = 1, repeatability, chunk additivity, argument errors, the host
mirror (Atmosphere.columnFluxes) and the full-size cfg4 column."""
import numpy as np
import pytest

from oracle import physics as ph
from oracle import ref_harness as rh
from pyrad_b200 import _lib
from pyrad_b200 import classes as C
from pyrad_b200 import distributed as pd
from pyrad_b200 import engine as eng
from pyrad_b200 import synth
from pyrad_b200 import workloads
from tests import flux_oracle as FO
from tests import golden_util as G
from tests import helpers as H

pytestmark = pytest.mark.gpu

ROWS_RTOL = 2e-5
FLUX_RTOL = 2e-5
FLUX_FLOOR = 1e-7            # of pi * integral B(T_surface)


def small_column(L):
    """A column at a small size: 1 layer runs K2's fused epilogue, 3 layers k3_fold_f32, 8 and 24 layers k3_fold_tma."""
    return workloads.atmosphere(n_layers=L, n_lines=6000, rmin=600.0, rmax=640.0, res=0.001,
                                top_km=2.0 if L == 1 else 40.0)


def run_column(engine, w):
    sp = w["species"]
    win = [eng.window_len(c, w["res"]) for c in w["cutoff"]]
    qt = np.array([[s.q(T) for s in sp] for T in w["T"]])
    engine.atmosphere(w["depth_cm"], w["T"], w["P"], w["conc"], [s.molmass for s in sp], qt, [s.q296 for s in sp], win,
                      w["t_surface"], w["range_max"])


def device_kmatrix(engine, L, n):
    import torch
    p, ld = engine.atmosphere_kmatrix_dev()
    k = pd.device_tensor(p, L * ld).view(L, ld)[:, :n]
    torch.cuda.synchronize()
    return k.cpu().numpy().astype(np.float64)


def quadrature(seed, n_mu):
    rng = np.random.default_rng(seed)
    return rng.uniform(0.1, 1.0, 4)[:n_mu], rng.uniform(0.05, 0.5, 4)[:n_mu]


def pi_int_planck(w):
    return ph.integrate_spectrum(ph.planck_wavenumber(ph.x_axis(w["range_min"], w["range_max"], w["res"]), w["t_surface"]),
                                 ph.pi, w["res"])


def check_fluxes(w, got, ref):
    up, down, ru, rd = got
    r_up, r_down, r_ru, r_rd = ref
    nu = ph.x_axis(w["range_min"], w["range_max"], w["res"])
    ok = nu > 0
    np.testing.assert_allclose(ru[:, ok], r_ru[:, ok], rtol=ROWS_RTOL)
    np.testing.assert_allclose(rd[:, ok], r_rd[:, ok], rtol=ROWS_RTOL)
    floor = FLUX_FLOOR * pi_int_planck(w)
    for a, b in ((up, r_up), (down, r_down)):
        err = np.abs(a - b)
        assert np.all(err <= FLUX_RTOL * np.abs(b) + floor), (err / np.maximum(np.abs(b), floor)).max()


@pytest.mark.parametrize("L", [1, 3, 8, 24])
def test_fluxes_match_the_fp64_fold_of_the_device_k_matrix(engine, L):
    w = small_column(L)
    n = H.engine_setup(engine, w)
    run_column(engine, w)
    if L == 1:
        assert engine.atmosphere_launches() == 2                  # K1 + K2 with the fused epilogue, no fold kernel
    k = device_kmatrix(engine, L, n)
    nu = ph.x_axis(w["range_min"], w["range_max"], w["res"])
    for n_mu in (1, 2, 3, 4):
        mu, wt = quadrature(100 + L, n_mu)
        got = engine.atmosphere_fluxes(mu, wt, rows=True)
        assert got[0].shape == got[1].shape == (L + 1,) and got[2].shape == got[3].shape == (n_mu, n)
        check_fluxes(w, got, FO.column_fluxes(k, w["depth_cm"], w["T"], w["t_surface"], nu, w["res"], mu, wt))


def test_fluxes_match_the_fp64_fold_of_the_oracle_k(engine):
    """The 8-layer column against k from the oracle's own line sums (as test_atmosphere_small)."""
    w = small_column(8)
    H.engine_setup(engine, w)
    run_column(engine, w)
    sp = w["species"]
    k = []
    for l in range(8):
        sig = H.oracle_sigma_groups(w, T=w["T"][l], P=w["P"][l], conc=w["conc"][l], cutoff=w["cutoff"][l])
        k.append(sum(ph.abs_coef(sig[g], w["conc"][l][g], w["P"][l], w["T"][l]) for g in range(len(sp))))
    nu = ph.x_axis(w["range_min"], w["range_max"], w["res"])
    for n_mu in (1, 4):
        mu, wt = quadrature(7, n_mu)
        got = engine.atmosphere_fluxes(mu, wt, rows=True)
        check_fluxes(w, got, FO.column_fluxes(k, w["depth_cm"], w["T"], w["t_surface"], nu, w["res"], mu, wt))


@pytest.mark.parametrize("L,tma", [(1, 1), (3, 1), (8, 1), (8, 0)])
def test_vertical_node_reproduces_the_column_radiance_bit_for_bit(engine, L, tma):
    w = small_column(L)
    n = H.engine_setup(engine, w)
    engine.set_option(eng.OPT_FOLD_TMA, tma)
    try:
        run_column(engine, w)
        up, _, ru, _ = engine.atmosphere_fluxes([1.0], [0.5], rows=True)
    finally:
        engine.set_option(eng.OPT_FOLD_TMA, 1)
    rad = np.empty(n, dtype=np.float32)
    engine.atmosphere_read_f32(rad, None)
    np.testing.assert_array_equal(ru[0], rad)
    # the W m-2 figure of PyRad's plotSpectrum legend: integrateSpectrum(radiance, pi)
    assert up[L] == pytest.approx(engine.atmosphere_integrate(np.pi, w["res"])[0], rel=1e-6)


def test_repeated_calls_give_identical_bits(engine):
    w = small_column(24)
    H.engine_setup(engine, w)
    run_column(engine, w)
    mu, wt = quadrature(3, 3)
    a = engine.atmosphere_fluxes(mu, wt, rows=True)
    b = engine.atmosphere_fluxes(mu, wt, rows=True)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


def test_chunks_add_up_to_the_whole_grid(engine):
    """Two tile-aligned chunks on one engine: the k matrix is shard invariant, so the rows concatenate bit for bit and
    the chunks' level fluxes add up to the whole grid's (only the FP64 order of the CTA sums differs)."""
    w = small_column(24)
    n = H.engine_setup(engine, w)
    mu, wt = quadrature(5, 3)
    run_column(engine, w)
    full = engine.atmosphere_fluxes(mu, wt, rows=True)
    parts = []
    for a, b in ((0, 16384), (16384, n)):
        H.engine_setup(engine, w, a, b)
        run_column(engine, w)
        parts.append(engine.atmosphere_fluxes(mu, wt, rows=True))
    for r in (2, 3):
        np.testing.assert_array_equal(np.concatenate([p[r] for p in parts], axis=1), full[r])
    for f in (0, 1):
        np.testing.assert_allclose(parts[0][f] + parts[1][f], full[f], rtol=1e-12, atol=0)


def test_argument_and_state_errors(engine):
    with eng.Engine(0) as fresh:
        with pytest.raises(_lib.EngineError) as ei:
            fresh.atmosphere_fluxes([1.0], [0.5])
        assert ei.value.code == -3                                  # PRB_ERR_STATE: no column yet
    w = small_column(3)
    H.engine_setup(engine, w)
    run_column(engine, w)
    bad = [([], []), ([0.5] * 5, [0.1] * 5), ([0.0], [0.5]), ([-0.5], [0.5]), ([1.5], [0.5]), ([0.5], [0.0]),
           ([0.5], [-1.0]), ([np.nan], [0.5]), ([0.5], [np.nan]), ([0.5, np.nan], [0.2, 0.3])]
    for mu, wt in bad:
        with pytest.raises(_lib.EngineError) as ei:
            engine.atmosphere_fluxes(mu, wt)
        assert ei.value.code == -2, (mu, wt)                        # PRB_ERR_ARG
    up, down = engine.atmosphere_fluxes([0.5], [1.0])               # and the engine still works
    assert np.all(np.isfinite(up)) and np.all(down[:-1] > 0) and down[-1] == 0


@pytest.fixture()
def data_root(tmp_path, engine):
    C.set_engine(engine)
    C.DATA_ROOT = str(tmp_path)
    C.Layer.hasAtmosphere = False
    old = C.BASE_RESOLUTION
    yield str(tmp_path)
    C.BASE_RESOLUTION = old
    C.DATA_ROOT = None


def test_host_mirror_column_fluxes(data_root):
    """Atmosphere.columnFluxes on a data tree (as tests/test_gpu_golden.py builds one): mu = 1, w = 1/2 gives the
    radiance of columnSpectrum bit for bit, and the heating rates are heatingRate of the returned fluxes."""
    g = G.load("cell_fine_grid")
    species = [str(s) for s in g["species"]]
    for i, s in enumerate(species):
        sp = synth.species(s)
        ln = G.lines_of(g, i)
        rh.write_params(data_root, sp.global_iso, sp.name, sp.mol_id, 1, 0.99, sp.q296, 1, sp.molmass)
        rh.write_q_table(data_root, sp.global_iso, range(100, 501), [sp.q(t) for t in range(100, 501)])
        rh.write_line_segments(data_root, sp.global_iso, sp.mol_id, 1, ln, int(ln["nu"].min() / 100) * 100,
                               ln["nu"].max() + 101)
    C.BASE_RESOLUTION = float(g["base"])
    atm = C.Atmosphere("column")
    rmin, rmax = float(g["range_min"]), float(g["range_max"])
    for depth, T, P in ((2e4, 280, 800.0), (3e4, 250, 300.0), (5e4, 220, 40.0), (8e4, 230, 3.0)):
        layer = atm.addLayer(depth, T, P, rmin, rmax, dynamicResolution=False)
        for s, c in zip(species, g["conc"]):
            layer.addMolecule(s, concentration=float(c))
    rad, _ = atm.columnSpectrum(288)
    out = atm.columnFluxes(288, mu=[1.0], weights=[0.5])
    np.testing.assert_array_equal(out["rad_up_top"][0].astype(np.float64), rad)
    np.testing.assert_array_equal(out["heating_rate"], C.heatingRate(out["flux_up"], out["flux_down"],
                                                                     [l.depth for l in atm], [l.T for l in atm],
                                                                     [l.P for l in atm]))
    np.testing.assert_array_equal(out["net"], out["flux_up"] - out["flux_down"])
    d = atm.columnFluxes(288)                                       # default: 3-node Gauss-Legendre on [0, 1]
    assert d["mu"].shape == (3,) and abs(np.sum(d["weights"] * d["mu"]) - 0.5) < 1e-15
    assert d["flux_up"].shape == (5,) and d["heating_rate"].shape == (4,) and d["rad_down_surface"].shape[0] == 3
    assert d["flux_down"][-1] == 0 and np.all(d["flux_down"][:-1] > 0) and np.all(d["flux_up"] > 0)


def test_cfg4_full_size_fluxes_with_the_default_quadrature(engine):
    """The 100-layer, 5 M-line, 5 M-point cfg4 column with 3 Gauss-Legendre nodes against an FP64 fold of the device's
    k matrix over the whole grid.  The oracle's formulas (tests/flux_oracle.py: Layer.transmission along the slant
    path, integrateSpectrum's sum) are evaluated here in blocks of grid points with torch float64 ON THE DEVICE -- the
    numpy restatement would take hours at this size; values beyond the FP32 range count as 0 as in flux_oracle.  Rows
    are compared at >= 1000 boundary-inclusive points, away from the few points next to 0 cm-1 where k < 0."""
    import torch
    w = workloads.atmosphere()
    n = H.engine_setup(engine, w)
    L = len(w["T"])
    assert n == 5_000_000 and L == 100
    run_column(engine, w)
    mu, wt = FO.gauss_legendre_01(3)
    up, down, ru, rd = engine.atmosphere_fluxes(mu, wt, rows=True)
    p, ld = engine.atmosphere_kmatrix_dev()
    kmat = pd.device_tensor(p, L * ld).view(L, ld)
    x0, dx, x_last, _ = eng.linspace_axis(w["range_min"], w["range_max"], n)
    h, c, kb = ph.h, ph.c, ph.k
    flt_max = float(np.finfo(np.float32).max)
    depth = [float(d) for d in w["depth_cm"]]
    r_up, r_down = np.zeros(L + 1), np.zeros(L + 1)
    pts = H.boundary_points(n, 1000, 91)
    assert len(pts) >= 1000
    ref_ru, ref_rd = np.zeros((3, len(pts))), np.zeros((3, len(pts)))
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
            sel = (pts >= a) & (pts < b)
            loc = torch.as_tensor(pts[sel] - a, device="cuda")

            def level_sum(I):
                return float(torch.where(I.abs() <= flt_max, I, torch.zeros_like(I)).sum())

            for i in range(3):
                f = 2 * ph.pi * wt[i] * mu[i] * w["res"]
                I = planck(w["t_surface"])
                r_up[0] += f * level_sum(I)
                for l in range(L):
                    t = torch.exp(-k[l] * depth[l] / mu[i])
                    I = t * I + (1 - t) * B[l]
                    r_up[l + 1] += f * level_sum(I)
                ref_ru[i, sel] = I[loc].cpu().numpy()
                I = torch.zeros_like(nu)
                for l in range(L - 1, -1, -1):
                    t = torch.exp(-k[l] * depth[l] / mu[i])
                    I = t * I + (1 - t) * B[l]
                    r_down[l] += f * level_sum(I)
                ref_rd[i, sel] = I[loc].cpu().numpy()
        kneg = (kmat[:, torch.as_tensor(pts, device="cuda")] < 0).any(dim=0).cpu().numpy()
    floor = FLUX_FLOOR * pi_int_planck(w)
    for name, a_, b_ in (("up", up, r_up), ("down", down, r_down)):
        err = np.abs(a_ - b_) / np.maximum(np.abs(b_), floor)
        assert err.max() <= FLUX_RTOL, (name, err.max(), int(err.argmax()), a_[int(err.argmax())], b_[int(err.argmax())])
    xa = x0 + pts * dx
    ok = ~kneg & (xa > 0)
    assert ok.sum() >= 990
    np.testing.assert_allclose(ru[:, pts][:, ok], ref_ru[:, ok], rtol=ROWS_RTOL)
    np.testing.assert_allclose(rd[:, pts][:, ok], ref_rd[:, ok], rtol=ROWS_RTOL)
    assert 150 < up[-1] < 400 and down[-1] == 0 and down[0] > 0     # W m-2 of an opaque 0-5000 cm-1 column
