"""GPU tests of the layer kernels (prb_atmosphere_save_base, prb_atmosphere_layer_kernels -> k3_kernel_base,
k3_kernel_tma, k3_flux_band_sum): the device against the FP64 O(L) formula (tests/kernel_oracle.py) over the engine's own
k matrices, against brute force on the device, the exactness rules, chunks, the base's state rules, the host mirror
(Atmosphere.columnKernels) and the full-size cfg4 column."""
import ctypes

import numpy as np
import pytest

from oracle import physics as ph
from pyrad_b200 import _lib
from pyrad_b200 import classes as C
from pyrad_b200 import distributed as pd
from pyrad_b200 import engine as eng
from pyrad_b200 import workloads
from tests import flux_oracle as FO
from tests import helpers as H
from tests import kernel_oracle as KO
from tests.test_gpu_band_fluxes import RRTMG_LW, axis, edge_sets
from tests.test_gpu_fluxes import data_root, device_kmatrix, quadrature, run_column, small_column  # noqa: F401

pytestmark = pytest.mark.gpu

#: |dev - oracle| <= KERNEL_RTOL * A + floor, A the magnitudes the FP32 operations round (kernel_oracle.layer_kernels)
KERNEL_RTOL = 2e-5
KERNEL_FLOOR = 1e-10        # of pi * the band's integral of B(T_surface)
KNEG_FLOOR = 1e-7           # of pi * the whole axis's integral of B(T_surface), for a band holding a point with k < 0


def perturb(w, kind):
    """The current column of a kind of perturbation: every layer +1 K or +0.01 K, 10 % or 1e-5 more depth, or 10 % more
    of the first gas (a different k row)."""
    if kind == "warm":
        return dict(w, T=w["T"] + 1.0, t_surface=w["t_surface"] + 1.0)
    if kind == "tiny":
        return dict(w, T=w["T"] + 0.01, t_surface=w["t_surface"] + 0.01)
    if kind == "depth":
        return dict(w, depth_cm=w["depth_cm"] * 1.1)
    if kind == "tiny_depth":
        return dict(w, depth_cm=w["depth_cm"] * (1 + 1e-5))
    conc = np.array(w["conc"], dtype=np.float64)
    conc[:, 0] *= 1.1
    return dict(w, conc=conc)


def column_state(w, k):
    return {"k": k, "depth_cm": np.asarray(w["depth_cm"], dtype=np.float64), "T": np.asarray(w["T"], dtype=np.float64),
            "t_surface": float(w["t_surface"])}


def floors(w, nu, edges, k_list):
    idx = np.searchsorted(edges, nu, side="right") - 1
    sel = (idx >= 0) & (idx < len(edges) - 1)
    b = np.nan_to_num(ph.planck_wavenumber(nu, w["t_surface"]))
    f = KERNEL_FLOOR * ph.pi * np.bincount(idx[sel], weights=b[sel], minlength=len(edges) - 1) * w["res"]
    neg = np.zeros(nu.size, dtype=bool)
    for k in k_list:
        neg |= (np.asarray(k) < 0).any(axis=0)
    hit = np.bincount(idx[sel & neg], minlength=len(edges) - 1) > 0
    return np.where(hit, KNEG_FLOOR * ph.pi * b.sum() * w["res"], f)


def check_kernels(got, ref, floor):
    worst = 0.0
    for g, r, a in ((got[0], ref[0], ref[2]), (got[1], ref[1], ref[3])):
        assert g.shape == r.shape
        tol = KERNEL_RTOL * a + floor[:, None]
        err = np.abs(g - r)
        assert np.all(err <= tol), (np.argwhere(err > tol)[:5], (err / np.maximum(tol, 1e-300)).max())
        worst = max(worst, float((err / np.maximum(tol, 1e-300)).max()))
    return worst


def base_and_current(engine, w, w2, n):
    L = len(w["T"])
    run_column(engine, w)
    kb = device_kmatrix(engine, L, n)
    engine.save_column_base()
    run_column(engine, w2)
    kc = device_kmatrix(engine, L, n)
    return column_state(w, kb), column_state(w2, kc)


@pytest.mark.parametrize("L", [1, 3, 8, 24])
@pytest.mark.parametrize("kind", ["warm", "depth", "conc", "tiny", "tiny_depth"])
def test_kernels_match_the_fp64_formula_over_the_device_k_matrices(engine, L, kind):
    w = small_column(L)
    n = H.engine_setup(engine, w)
    w2 = perturb(w, kind)
    base, cur = base_and_current(engine, w, w2, n)
    nu = axis(w)
    sets = edge_sets(nu, L)
    names = ["1_and_3_points", "127_128_129_points", "random", "whole"] if kind != "warm" else list(sets)
    for n_mu in (1, 2, 3, 4):
        mu, wt = quadrature(500 + L, n_mu)
        for name in names:
            edges = sets[name]
            got = engine.atmosphere_layer_kernels(mu, wt, edges)
            assert got[0].shape == got[1].shape == (len(edges) - 1, L + 1), name
            ref = KO.layer_kernels(base, cur, nu, w["res"], mu, wt, edges)
            check_kernels(got, ref, floors(w, nu, edges, [base["k"], cur["k"]]))
            assert np.all(got[1][:, 0] == 0)


@pytest.mark.parametrize("rmin", [0.0, 4960.0])
def test_kernels_on_grids_at_zero_and_high_wavenumber(engine, rmin):
    w = workloads.atmosphere(n_layers=8, n_lines=6000, rmin=rmin, rmax=rmin + 40.0, res=0.001, top_km=40.0)
    n = H.engine_setup(engine, w)
    base, cur = base_and_current(engine, w, perturb(w, "warm"), n)
    nu = axis(w)
    edges = np.concatenate([[rmin], np.sort(np.random.default_rng(3).uniform(rmin, rmin + 40, 9)), [rmin + 41]])
    for n_mu in (1, 3):
        mu, wt = FO.gauss_legendre_01(n_mu)
        got = engine.atmosphere_layer_kernels(mu, wt, edges)
        check_kernels(got, KO.layer_kernels(base, cur, nu, w["res"], mu, wt, edges),
                      floors(w, nu, edges, [base["k"], cur["k"]]))


def test_a_warm_top_is_the_same_start_for_both_columns(engine):
    w = small_column(8)
    n = H.engine_setup(engine, w)
    base, cur = base_and_current(engine, w, perturb(w, "warm"), n)
    nu = axis(w)
    mu, wt = FO.gauss_legendre_01(3)
    edges = edge_sets(nu, 1)["random"]
    engine.set_flux_boundaries(t_top=250.0)
    try:
        got = engine.atmosphere_layer_kernels(mu, wt, edges)
    finally:
        engine.set_flux_boundaries()
    check_kernels(got, KO.layer_kernels(base, cur, nu, w["res"], mu, wt, edges, t_top=250.0),
                  floors(w, nu, edges, [base["k"], cur["k"]]))
    plain = engine.atmosphere_layer_kernels(mu, wt, edges)
    assert got[0].tobytes() == plain[0].tobytes()                     # the upward pass does not see the top


@pytest.mark.parametrize("layer", [0, 5, 23])
def test_kernels_equal_brute_force_on_the_device(engine, layer):
    """Only layer l warmer: every other row is the base's bit for bit, and the band flux calls' difference agrees with
    entry l + 1 within the rounding of the two FP32 flux calls: 2e-6 of each band's flux (the level sums of a call
    are good to ~1e-6 of F) plus the kernels' own KERNEL_RTOL * A."""
    w = small_column(24)
    n = H.engine_setup(engine, w)
    L = 24
    mu, wt = FO.gauss_legendre_01(3)
    edges = np.array([600.0, 610.0, 625.0, 641.0])
    run_column(engine, w)
    kb = device_kmatrix(engine, L, n)
    fb = engine.atmosphere_band_fluxes(mu, wt, edges)
    engine.save_column_base()
    T = w["T"].copy()
    T[layer] += 1.0
    w2 = dict(w, T=T)
    run_column(engine, w2)
    kc = device_kmatrix(engine, L, n)
    others = [m for m in range(L) if m != layer]
    assert kc[others].tobytes() == kb[others].tobytes()
    fc = engine.atmosphere_band_fluxes(mu, wt, edges)
    up, down = engine.atmosphere_layer_kernels(mu, wt, edges)
    ref = KO.layer_kernels(column_state(w, kb), column_state(w2, kc), axis(w), w["res"], mu, wt, edges)
    d_up, d_down = fc[0][:, L] - fb[0][:, L], fc[1][:, 0] - fb[1][:, 0]
    tol_up = 2e-6 * np.abs(fb[0][:, L]) + KERNEL_RTOL * ref[2][:, layer + 1]
    tol_down = 2e-6 * np.abs(fb[1][:, 0]) + KERNEL_RTOL * ref[3][:, layer + 1]
    assert np.all(np.abs(d_up - up[:, layer + 1]) <= tol_up), (d_up, up[:, layer + 1])
    assert np.all(np.abs(d_down - down[:, layer + 1]) <= tol_down), (d_down, down[:, layer + 1])
    assert np.all(up[:, [m + 1 for m in others]] == 0) and np.all(down[:, [m + 1 for m in others]] == 0)
    assert np.all(up[:, 0] == 0)


def test_the_same_column_again_gives_zeros_and_repeated_calls_the_same_bits(engine):
    w = small_column(24)
    H.engine_setup(engine, w)
    run_column(engine, w)
    engine.save_column_base()
    run_column(engine, w)
    mu, wt = FO.gauss_legendre_01(3)
    edges = edge_sets(axis(w), 2)["random"]
    for x in engine.atmosphere_layer_kernels(mu, wt, edges):
        assert np.all(x == 0) and not np.any(np.signbit(x))
    run_column(engine, perturb(w, "warm"))
    a = engine.atmosphere_layer_kernels(mu, wt, edges)
    b = engine.atmosphere_layer_kernels(mu, wt, edges)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
    assert np.any(a[0] != 0)


def _chunk_kernels(engine, w, w2, lo, hi, mu, wt, edges):
    n = eng.grid_len(w["range_min"], w["range_max"], w["res"])
    engine.set_grid(w["range_min"], w["res"], n, lo, hi)
    run_column(engine, w)
    engine.save_column_base()
    run_column(engine, w2)
    return engine.atmosphere_layer_kernels(mu, wt, edges)


def test_chunks_give_their_bands_bit_for_bit_and_add_up_to_the_whole_grid(engine):
    w = small_column(8)
    n = H.engine_setup(engine, w)
    w2 = perturb(w, "warm")
    nu = axis(w)
    mu, wt = FO.gauss_legendre_01(3)
    inside = np.array([nu[200], nu[5000], nu[16000]])                 # both bands inside the first chunk
    edges = np.concatenate([[nu[0]], np.sort(np.random.default_rng(5).uniform(nu[0], nu[-1], 40)), [nu[-1] + 1]])
    whole_in = _chunk_kernels(engine, w, w2, 0, n, mu, wt, inside)
    whole = engine.atmosphere_layer_kernels(mu, wt, edges)
    part_in = _chunk_kernels(engine, w, w2, 0, 16384, mu, wt, inside)
    for x, y in zip(whole_in, part_in):
        assert x.tobytes() == y.tobytes()
    for cuts in ([0, 16384, n], [0, 16384, 32768, n]):
        acc = [np.zeros_like(whole[0]), np.zeros_like(whole[1])]
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            got = _chunk_kernels(engine, w, w2, lo, hi, mu, wt, edges)
            acc[0] += got[0]
            acc[1] += got[1]
        for x, y in zip(acc, whole):
            np.testing.assert_allclose(x, y, rtol=1e-12, atol=1e-12 * np.abs(y).max())


def _status(engine, mu=(0.5,), wt=(1.0,), edges=(600.0, 641.0)):
    m, w, e = (np.ascontiguousarray(x, dtype=np.float64) for x in (mu, wt, edges))
    dp = ctypes.POINTER(ctypes.c_double)
    out = np.zeros(64 * 1024)
    return engine._lib.prb_atmosphere_layer_kernels(engine._h, m.size, m.ctypes.data_as(dp), w.ctypes.data_as(dp),
                                                    e.size - 1, e.ctypes.data_as(dp), out.ctypes.data_as(dp),
                                                    out.ctypes.data_as(dp))


def test_state_rules(engine):
    w = small_column(3)
    n = H.engine_setup(engine, w)
    run_column(engine, w)
    assert _status(engine) == -3                                       # no base
    assert engine._lib.prb_atmosphere_save_base(engine._h) == 0
    assert _status(engine) == 0
    engine.set_grid(w["range_min"], w["res"], n)                       # the same grid: the base is dropped
    run_column(engine, w)
    assert _status(engine) == -3
    engine.save_column_base()
    sp = w["species"]
    qt = np.array([[s.q(T) for s in sp] for T in w["T"]])
    with pytest.raises(_lib.EngineError):                              # a failed column keeps the base ...
        engine.atmosphere(w["depth_cm"], w["T"], w["P"], w["conc"], [s.molmass for s in sp], qt, [s.q296 for s in sp],
                          [0, 0, 0], w["t_surface"], w["range_max"])
    assert _status(engine) == -3                                       # ... but leaves no current column
    run_column(engine, perturb(w, "warm"))                             # a new column keeps it
    assert _status(engine) == 0
    w4 = small_column(8)
    run_column(engine, dict(w4, lines=w["lines"]))                    # another layer count
    assert _status(engine) == -3
    run_column(engine, w)
    assert _status(engine) == 0
    engine.set_flux_boundaries(emissivity=0.9)
    assert _status(engine) == -3
    engine.set_flux_boundaries(t_top=3.0)                             # a warm top alone is allowed
    assert _status(engine) == 0
    engine.set_flux_boundaries()
    engine.set_solar_source(([500.0, 700.0], [1.0, 1.0]), 0.5)
    try:
        assert _status(engine) == -3
    finally:
        engine.set_solar_source()
    assert _status(engine) == 0
    for mu, wt, edges in (((0.0,), (1.0,), (600.0, 641.0)), ((0.5,) * 5, (1.0,) * 5, (600.0, 641.0)),
                          ((0.5,), (-1.0,), (600.0, 641.0)), ((0.5,), (1.0,), (641.0, 600.0)),
                          ((0.5,), (1.0,), (600.0, np.inf))):
        assert _status(engine, mu, wt, edges) == -2
    engine.peer_alloc(0, 1, n)                                         # a peer buffer: dropped
    run_column(engine, w)
    assert _status(engine) == -3
    engine.save_column_base()
    engine._lib.prb_peer_disconnect(engine._h)
    run_column(engine, w)
    assert _status(engine) == -3
    # prb_gas_cell_host sets its own grid
    H.engine_setup(engine, w)
    run_column(engine, w)
    engine.save_column_base()
    g = workloads.gas_cell(["co2", "h2o"], 4000, 600.0, 640.0, 0.001, 260, 800.0, [400e-6, 0.01], 10.0, 31)
    gs = g["species"]
    engine.gas_cell_host(g["lines"], len(gs), g["range_min"], g["res"], n, 0, n, g["depth_cm"], g["T"], g["P"],
                         g["conc"], [s.molmass for s in gs], [s.q(g["T"]) for s in gs], [s.q296 for s in gs],
                         eng.window_len(g["cutoff"], g["res"]), 288.0, g["range_max"])
    assert _status(engine) == -3


def test_host_mirror_column_kernels(data_root):
    """Atmosphere.columnKernels on a data tree against the oracle over the mirror's own k matrices, with and without a
    continuum; one band by default; and its argument checks that need layers."""
    from tests import continuum_oracle as CO
    from tests import golden_util as G
    from tests.test_gpu_band_fluxes import _column_on_data_tree
    atm, rmin, rmax = _column_on_data_tree(data_root)
    g = G.load("cell_fine_grid")
    warm = C.Atmosphere("warm")
    for l in atm:
        layer = warm.addLayer(l.depth, l.T + 1, l.P, rmin, rmax, dynamicResolution=False)
        for sname, c in zip([str(x) for x in g["species"]], g["conc"]):
            layer.addMolecule(sname, concentration=float(c))
    e = C.engine()
    mu, wt = FO.gauss_legendre_01(3)
    edges = np.linspace(rmin, rmax + 1.0, 5)
    L = len(atm)
    for continuum in (None, CO.synthetic_table(29, rmin - 5.0, rmax + 5.0, spacing=2.0)):
        out = atm.columnKernels(288.0, warm, 289.0, mu=mu, weights=wt, bands=edges, continuum=continuum)
        assert out["toa_up"].shape == out["surface_down"].shape == (4, L) and out["toa_up_surface"].shape == (4,)
        np.testing.assert_array_equal(out["band_edges"], edges)
        states = []
        for a, ts in ((atm, 288.0), (warm, 289.0)):
            ks = a._column(ts, lambda en: device_kmatrix(en, L, en.n_chunk), continuum)
            states.append({"k": ks, "depth_cm": [l.depth for l in a], "T": [float(l.T) for l in a], "t_surface": ts})
        nu = np.linspace(rmin, rmax, e.n_chunk)
        ref = KO.layer_kernels(states[0], states[1], nu, C.BASE_RESOLUTION, mu, wt, edges)
        got = (np.concatenate([out["toa_up_surface"][:, None], out["toa_up"]], axis=1),
               np.concatenate([np.zeros((4, 1)), out["surface_down"]], axis=1))
        check_kernels(got, ref, floors({"t_surface": 288.0, "res": C.BASE_RESOLUTION}, nu, edges,
                                       [states[0]["k"], states[1]["k"]]))
        assert np.all(out["toa_up"] >= 0) and np.any(out["toa_up"] > 0) and np.all(out["toa_up_surface"] >= 0)
    one = atm.columnKernels(288.0, warm, 289.0)
    assert one["toa_up"].shape == (1, L) and one["mu"].size == 3
    short = C.Atmosphere("short")
    short.addLayer(atm[0].depth, atm[0].T, atm[0].P, rmin, rmax, dynamicResolution=False)
    with pytest.raises(ValueError, match="layers"):
        atm.columnKernels(288.0, short)
    with pytest.raises(ValueError, match="bands"):
        atm.columnKernels(288.0, warm, bands=[rmax, rmin])
    dry = C.Atmosphere("one gas")                                     # another line list: refused
    for l in atm:
        layer = dry.addLayer(l.depth, l.T + 1, l.P, rmin, rmax, dynamicResolution=False)
        layer.addMolecule(str(g["species"][0]), concentration=float(g["conc"][0]))
    with pytest.raises(ValueError, match="line list"):
        atm.columnKernels(288.0, dry)


def test_cfg4_full_size_layer_kernels(engine):
    """The 100-layer, 5 M-point cfg4 column and a +1 K column with 3 Gauss-Legendre nodes, in RRTMG's 16 longwave bands
    and four more up to 5000 cm-1, against the O(L) formula restated in FP64 with torch on the device (per-band sums by
    index_add)."""
    import torch
    w = workloads.atmosphere()
    n = H.engine_setup(engine, w)
    L = len(w["T"])
    assert n == 5_000_000 and L == 100
    w2 = perturb(w, "warm")
    edges = np.array(RRTMG_LW + [3500.0, 4000.0, 4500.0, 5001.0])
    mu, wt = FO.gauss_legendre_01(3)
    run_column(engine, w)
    p, ld = engine.atmosphere_kmatrix_dev()
    kb_all = pd.device_tensor(p, L * ld).view(L, ld)[:, :n].clone()
    engine.save_column_base()
    run_column(engine, w2)
    got = engine.atmosphere_layer_kernels(mu, wt, edges)
    p, ld = engine.atmosphere_kmatrix_dev()
    kc_all = pd.device_tensor(p, L * ld).view(L, ld)[:, :n]
    x0, dx, x_last, _ = eng.linspace_axis(w["range_min"], w["range_max"], n)
    h, c, kB = ph.h, ph.c, ph.k
    db, Tb, Tc = [float(d) for d in w["depth_cm"]], [float(t) for t in w["T"]], [float(t) for t in w2["T"]]
    dc = [float(d) for d in w2["depth_cm"]]
    nb = len(edges) - 1
    ref = [torch.zeros(nb + 1, L + 1, dtype=torch.float64, device="cuda") for _ in range(4)]
    pib = torch.zeros(nb + 1, dtype=torch.float64, device="cuda")
    kneg = torch.zeros(nb + 1, dtype=torch.bool, device="cuda")
    et = torch.as_tensor(edges, device="cuda")
    block = 1 << 20
    with torch.no_grad():
        for a in range(0, n, block):
            b = min(n, a + block)
            nu = torch.arange(a, b, dtype=torch.float64, device="cuda") * dx + x0
            if b == n:
                nu[-1] = x_last

            def planck(T):
                return 2E8 * h * c ** 2 * nu ** 3 / (torch.exp(100 * h * c * nu / kB / T) - 1)

            def dplanck(T, T2):
                return planck(T) * torch.expm1(ph.c2 * nu * ((T2 - T) / (T * T2))) / -torch.expm1(-ph.c2 * nu / T2)

            i = torch.searchsorted(et, nu, right=True) - 1
            ids = torch.where((i >= 0) & (i < nb), i, torch.full_like(i, nb))
            kb, kc = kb_all[:, a:b].double(), kc_all[:, a:b].double()
            kneg[ids[((kb < 0) | (kc < 0)).any(dim=0)]] = True
            pib.index_add_(0, ids, torch.nan_to_num(planck(w["t_surface"])))
            tau = [kb[l] * db[l] for l in range(L)]
            dtau = [(kc[l] - kb[l]) * dc[l] + kb[l] * (dc[l] - db[l]) for l in range(L)]
            S = torch.stack(tau).sum(dim=0)
            B = [planck(T) for T in Tb]
            dB = [dplanck(T, T2) for T, T2 in zip(Tb, Tc)]

            def add(r, mag, j, f, cval, aval):
                ok = torch.isfinite(cval) & torch.isfinite(aval)
                ref[r][:, j].index_add_(0, ids, torch.where(ok, cval, torch.zeros_like(cval)) * f)
                ref[mag][:, j].index_add_(0, ids, torch.where(torch.isfinite(aval), aval, torch.zeros_like(aval)) * f)

            for m, wq in zip(mu, wt):
                f = 2 * ph.pi * wq * m * w["res"]
                dbs = dplanck(float(w["t_surface"]), float(w2["t_surface"]))
                u = torch.exp(-S / m)
                add(0, 2, 0, f, u * dbs, u * dbs.abs())
                for r, mag, order, I in ((0, 2, range(L), planck(w["t_surface"])),
                                         (1, 3, range(L - 1, -1, -1), torch.zeros_like(nu))):
                    rem = S.clone()
                    for l in order:
                        t = torch.exp(-tau[l] / m)
                        dt = KO.transmittance_difference(tau[l], dtau[l], m, xp=torch)
                        omt = -torch.expm1(-(tau[l] + dtau[l]) / m)
                        di = omt * dB[l] + dt * (I - B[l])
                        rem = rem - tau[l]
                        U = torch.exp(-rem / m)
                        add(r, mag, l + 1, f, U * di,
                            U * ((omt * dB[l]).abs() + dt.abs() * (I.abs() + B[l].abs())))
                        I = t * I + (1 - t) * B[l]
    ref_np = [x[:-1].cpu().numpy() for x in ref]
    floor = KERNEL_FLOOR * ph.pi * pib[:-1].cpu().numpy() * w["res"]
    total = KNEG_FLOOR * ph.pi * float(pib.sum()) * w["res"]
    floor = np.where(kneg[:-1].cpu().numpy(), total, floor)
    worst = check_kernels(got, ref_np, floor)
    print(f"cfg4 layer kernels: worst |dev - ora| / tol = {worst:.3g}")
    assert np.all(got[1][:, 0] == 0)
