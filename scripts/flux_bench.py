"""Time prb_atmosphere_fluxes on the cfg4 column (100 layers, ~5 M lines, 0-5000 cm-1 at 0.001 cm-1: 5 M points).

Runs the column once through prb_atmosphere (far-field K2, as bench.py's atmosphere object), times it, then times the
flux call for 1, 2, 3 and 4 angular nodes (Gauss-Legendre on [0, 1]) on the same resident k matrix: CUDA events on the
engine stream around each call (the layer-table upload, the upward and downward k3_flux_tma passes, the two k3_flux_sum
launches and the copy of the level fluxes), warm-up first, then --reps calls.  Also reports the algorithmic bytes (the
k matrix read once per pass, L N 4 bytes, two passes) and their rate against prb_measure_peaks' copy bandwidth, and the
device name and power limit read in the same run.  Then times prb_atmosphere_band_fluxes with 3 nodes on the same
k matrix, for four band sets -- one band over the whole grid, RRTMG's 16 longwave bands, 5000 bands of 1 cm-1 and the
single band 630-700 cm-1 -- and reports each beside the 3-node total call of the same run.  Last, with the flux
boundaries set (prb_set_flux_boundaries: emissivity 0.98 with a linear dip to 0.75 over 1080-1180 cm-1, the 2.725 K
cosmic background at the top, Lambertian and specular reflection), times the 3-node total call and the 16-band call as
ratios to the plain calls timed right before them, and reports the OLR and the net flux at the surface with and
without the surface.  Then, on the same surface and top, adds a 5772 K blackbody Sun scaled to 1361 W m-2 in total at
mu_sun = 0.5 (prb_set_solar_source, both reflections), times the same two calls as ratios to the sunless boundary calls
timed right before them, and reports the sunlight at the top (mu_sun sum S res), the beam at the surface, the sunlight
leaving the top and the largest solar heating rate with its layer, each as the result with the Sun minus the result
without it.  Last, a water-vapour continuum (prb_set_continuum) from a SYNTHETIC table in MT_CKD's form (seeded,
log-uniform coefficients, not MT_CKD's values) with cfg4's H2O profile: the column itself (prb_atmosphere) timed five
times without and five times with it, alternating, the median difference against the add kernel's algorithmic bytes
(the k matrix read and written once, 2 L N 4) and the copy bandwidth, and the change it makes to the OLR, the surface
down flux and RRTMG's 16 band fluxes (3 nodes).  Last, the layer kernels: prb_atmosphere_save_base on the plain column and
prb_atmosphere_layer_kernels (3 nodes, RRTMG's 16 bands) against a column 1 K warmer, each as a ratio to the 16-band
flux call timed right before it, and the OLR temperature kernel's column sum beside the OLR difference of the two
columns (they differ by the layers' non-additivity).  Prints one JSON line; writes nothing.

    python scripts/flux_bench.py [--reps 30] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_power():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20).stdout
        name, limit, mhz = [x.strip() for x in out.strip().splitlines()[0].split(",")]
        return {"nvidia_smi_name": name, "power_limit_w": float(limit), "sm_max_mhz": float(mhz)}
    except Exception as ex:                                   # the timing stands without it; say why it is missing
        return {"nvidia_smi_error": str(ex)}


def timed(stream, fn, warmup, reps):
    import torch
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return ms


def blackbody_sun(nu_t, t_sun=5772.0, total=1361.0):
    """A blackbody Sun scaled to `total` W m-2 over all wavenumbers, as an irradiance table (nu, S) on nu_t."""
    from oracle import physics as ph
    fine = np.arange(1.0, 100000.0, 1.0)
    scale = total / (ph.pi * np.sum(ph.planck_wavenumber(fine, t_sun)))
    return nu_t, ph.pi * np.nan_to_num(ph.planck_wavenumber(nu_t, t_sun)) * scale


def solar_section(e, stream, args, w, mu, wt, calls, eps_table):
    """The Sun on cfg4's surface (eps_table, 2.725 K top): both reflections, each timed right after the same sunless
    boundary calls."""
    from pyrad_b200.classes import heatingRate
    sun, mu_sun = blackbody_sun(np.arange(0.0, 5011.0)), 0.5
    res = {"t_sun_k": 5772.0, "total_w_m2": 1361.0, "mu_sun": mu_sun, "n_mu": 3, "runs": []}

    def heating(up, down):
        return heatingRate(up, down, w["depth_cm"], w["T"], w["P"])

    try:
        for reflection in ("lambertian", "specular"):
            e.set_flux_boundaries(eps_table, reflection, 2.725)
            e.set_solar_source()
            dark_ms = {k: float(np.median(timed(stream, f, args.warmup, args.reps))) for k, f in calls.items()}
            up0, down0 = e.atmosphere_fluxes(mu, wt)
            e.set_solar_source(sun, mu_sun)
            run = {"reflection": reflection, "sunless_ms_median": dark_ms}
            for k, f in calls.items():
                ms = timed(stream, f, args.warmup, args.reps)
                med = float(np.median(ms))
                run[k] = {"ms_median": med, "ms_p10_p90": [float(np.percentile(ms, 10)), float(np.percentile(ms, 90))],
                          "reps": args.reps, "ratio_to_sunless_call": med / dark_ms[k]}
            up, down = e.atmosphere_fluxes(mu, wt)
            dq = heating(up, down) - heating(up0, down0)
            run.update(sun_top_w_m2=float(down[-1] - down0[-1]), beam_surface_w_m2=float(down[0] - down0[0]),
                       sun_leaving_top_w_m2=float(up[-1] - up0[-1]), max_solar_heating_k_day=float(dq.max()),
                       max_solar_heating_layer=int(dq.argmax()), max_solar_heating_p_hpa=float(w["P"][int(dq.argmax())]))
            res["runs"].append(run)
    finally:
        e.set_solar_source()
        e.set_flux_boundaries()
    return res


def synthetic_continuum(seed=4, lo=0.0, hi=5000.0, spacing=10.0):
    """A table in MT_CKD's form, NOT MT_CKD's values: coefficients log-uniform in [1e-27, 1e-21] cm2 molecule-1 (cm-1)-1,
    exponents uniform in [0, 6], entries `spacing` cm-1 apart (tests/continuum_oracle.synthetic_table)."""
    rng = np.random.default_rng(seed)
    m = int(round((hi - lo) / spacing)) + 1
    return {"nu": np.linspace(lo, hi, m), "self": 10.0 ** rng.uniform(-27, -21, m),
            "foreign": 10.0 ** rng.uniform(-27, -21, m), "texp": rng.uniform(0.0, 6.0, m)}


def continuum_section(e, stream, w, column, mu, wt, rrtmg, copy_bytes_per_s, runs=5):
    """The column with and without the continuum, alternating; then what the continuum changes in the 3-node fluxes."""
    table, x = synthetic_continuum(), np.asarray(w["conc"])[:, 0]
    L, n = len(w["T"]), e.n_chunk

    def fluxes():
        up, down = e.atmosphere_fluxes(mu, wt)
        bu, bd = e.atmosphere_band_fluxes(mu, wt, rrtmg)
        return up, down, bu, bd

    plain, wet = [], []
    try:
        for i in range(runs):
            e.set_continuum()
            plain += timed(stream, column, 1 if i == 0 else 0, 1)
            e.set_continuum(table, x)
            wet += timed(stream, column, 1 if i == 0 else 0, 1)
        wet_f = fluxes()
        e.set_continuum()
        column()
        dry_f = fluxes()
    finally:
        e.set_continuum()
    diff = float(np.median(wet) - np.median(plain))
    add_bytes = 2 * L * n * 4
    return {"table": "synthetic (seeded, log-uniform 1e-27..1e-21, t_exp 0..6, 10 cm-1 spacing over 0-5000 cm-1; "
                     "not MT_CKD)", "mole_fraction": "cfg4 H2O profile", "runs": runs,
            "plain_ms": plain, "continuum_ms": wet, "plain_ms_median": float(np.median(plain)),
            "continuum_ms_median": float(np.median(wet)), "median_difference_ms": diff,
            "add_bytes": add_bytes, "add_ms_at_copy_bandwidth": add_bytes / copy_bytes_per_s * 1e3,
            "olr_change_w_m2": float(wet_f[0][-1] - dry_f[0][-1]),
            "surface_down_change_w_m2": float(wet_f[1][0] - dry_f[1][0]),
            "rrtmg_band_edges": [float(v) for v in rrtmg],
            "band_olr_change_w_m2": [float(v) for v in wet_f[2][:, -1] - dry_f[2][:, -1]],
            "band_surface_down_change_w_m2": [float(v) for v in wet_f[3][:, 0] - dry_f[3][:, 0]]}


def kernels_section(e, stream, args, w, column, mu, wt, rrtmg):
    """prb_atmosphere_save_base and prb_atmosphere_layer_kernels (3 nodes, RRTMG's 16 bands) on the plain column and a
    column 1 K warmer in every layer and at the surface, each timed as a ratio to the 16-band flux call timed right before
    it; then the OLR temperature kernel's column sum beside the OLR difference of the two columns."""
    from pyrad_b200 import engine as eng
    sp = w["species"]
    win = [eng.window_len(c, w["res"]) for c in w["cutoff"]]
    t_warm = np.asarray(w["T"]) + 1.0
    warm = e.atmosphere_call(w["depth_cm"], t_warm, w["P"], w["conc"], [s.molmass for s in sp],
                             np.array([[s.q(T) for s in sp] for T in t_warm]), [s.q296 for s in sp], win,
                             w["t_surface"] + 1.0, w["range_max"])
    band = lambda: e.atmosphere_band_fluxes(mu, wt, rrtmg)                      # noqa: E731
    column()
    up0, _ = e.atmosphere_fluxes(mu, wt)

    def stats(ms):
        return {"ms_median": float(np.median(ms)), "ms_p10_p90": [float(np.percentile(ms, 10)),
                                                                  float(np.percentile(ms, 90))], "reps": args.reps}
    band_a = stats(timed(stream, band, args.warmup, args.reps))
    save = stats(timed(stream, e.save_column_base, args.warmup, args.reps))
    warm()
    up1, _ = e.atmosphere_fluxes(mu, wt)
    band_b = stats(timed(stream, band, args.warmup, args.reps))
    kern = stats(timed(stream, lambda: e.atmosphere_layer_kernels(mu, wt, rrtmg), args.warmup, args.reps))
    toa, sfc = e.atmosphere_layer_kernels(mu, wt, rrtmg)
    out = {"n_mu": 3, "bands": "rrtmg_lw_16", "perturbation": "+1 K in every layer and at the surface",
           "band_call_before_save": band_a, "save_base": save,
           "save_base_ratio_to_band_call": save["ms_median"] / band_a["ms_median"],
           "band_call_before_kernels": band_b, "layer_kernels": kern,
           "layer_kernels_ratio_to_band_call": kern["ms_median"] / band_b["ms_median"],
           "olr_kernel_column_sum_w_m2": float(toa.sum()),
           "olr_kernel_layers_w_m2": float(toa[:, 1:].sum()), "olr_kernel_surface_w_m2": float(toa[:, 0].sum()),
           "olr_difference_of_the_columns_w_m2": float(up1[-1] - up0[-1]),
           "surface_down_kernel_column_sum_w_m2": float(sfc.sum())}
    column()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--atm-reps", type=int, default=5)
    args = ap.parse_args()
    if args.reps < 20:
        ap.error("--reps must be at least 20")
    import torch
    from pyrad_b200 import engine as eng
    from pyrad_b200 import workloads

    if not torch.cuda.is_available():
        raise SystemExit("flux_bench: no CUDA device (there is no CPU measurement)")
    w = workloads.atmosphere()
    sp = w["species"]
    L = len(w["T"])
    e = eng.Engine(0)
    n = eng.grid_len(w["range_min"], w["range_max"], w["res"])
    e.upload_lines(w["lines"], n_groups=len(sp))
    e.set_grid(w["range_min"], w["res"], n)
    win = [eng.window_len(c, w["res"]) for c in w["cutoff"]]
    qt = np.array([[s.q(T) for s in sp] for T in w["T"]])
    column = e.atmosphere_call(w["depth_cm"], w["T"], w["P"], w["conc"], [s.molmass for s in sp], qt,
                               [s.q296 for s in sp], win, w["t_surface"], w["range_max"])
    stream = torch.cuda.ExternalStream(e.stream)
    e.set_k2_variant(eng.K2_FARFIELD, 0)
    atm_ms = timed(stream, column, 1, args.atm_reps)
    peaks = e.measure_peaks()
    pass_bytes = L * n * 4
    out = {"workload": "cfg4: %d layers, %d lines, %d points, far-field K2" % (L, len(w["lines"]["nu"]), n),
           "device": torch.cuda.get_device_name(0), **device_power(),
           "atmosphere_ms_median": float(np.median(atm_ms)), "atmosphere_ms_runs": atm_ms,
           "copy_bytes_per_s": peaks["copy_bytes_per_s"], "kmatrix_pass_bytes": pass_bytes, "fluxes": []}
    for n_mu in (1, 2, 3, 4):
        x, wt = np.polynomial.legendre.leggauss(n_mu)
        mu, wt = (x + 1) / 2, wt / 2
        ms = timed(stream, lambda: e.atmosphere_fluxes(mu, wt), args.warmup, args.reps)
        med = float(np.median(ms))
        up, down = e.atmosphere_fluxes(mu, wt)
        out["fluxes"].append({
            "n_mu": n_mu, "ms_median": med, "ms_min": float(np.min(ms)), "ms_max": float(np.max(ms)),
            "ms_p10_p90": [float(np.percentile(ms, 10)), float(np.percentile(ms, 90))], "reps": args.reps,
            "bytes_per_s": 2 * pass_bytes / (med * 1e-3),
            "share_of_copy_bandwidth": 2 * pass_bytes / (med * 1e-3) / peaks["copy_bytes_per_s"],
            "share_of_atmosphere": med / float(np.median(atm_ms)),
            "olr_w_m2": float(up[-1]), "surface_down_w_m2": float(down[0])})
    x, wt = np.polynomial.legendre.leggauss(3)
    mu, wt = (x + 1) / 2, wt / 2
    total_ms = next(f["ms_median"] for f in out["fluxes"] if f["n_mu"] == 3)
    band_sets = {"whole_grid": [w["range_min"], w["range_max"] + w["res"]],
                 "rrtmg_lw_16": [10, 350, 500, 630, 700, 820, 980, 1080, 1180, 1390, 1480, 1800, 2080, 2250, 2380,
                                 2600, 3250],
                 "one_cm_5000": np.arange(0.0, 5001.0),
                 "co2_630_700": [630.0, 700.0]}
    out["band_fluxes"] = []
    for name, edges in band_sets.items():
        edges = np.asarray(edges, dtype=np.float64)
        ms = timed(stream, lambda: e.atmosphere_band_fluxes(mu, wt, edges), args.warmup, args.reps)
        med = float(np.median(ms))
        bu, _ = e.atmosphere_band_fluxes(mu, wt, edges)
        out["band_fluxes"].append({
            "bands": name, "n_bands": len(edges) - 1, "n_mu": 3, "ms_median": med,
            "ms_p10_p90": [float(np.percentile(ms, 10)), float(np.percentile(ms, 90))], "reps": args.reps,
            "ratio_to_total_call": med / total_ms, "olr_w_m2": float(bu[:, -1].sum())})
    # boundaries: a grey surface with a reststrahlen-like dip and the cosmic background at the top
    eps_table = ([1080.0, 1130.0, 1180.0], [0.98, 0.75, 0.98])
    rrtmg = np.asarray(band_sets["rrtmg_lw_16"], dtype=np.float64)
    calls = {"total": lambda: e.atmosphere_fluxes(mu, wt), "rrtmg_lw_16": lambda: e.atmosphere_band_fluxes(mu, wt, rrtmg)}
    e.set_flux_boundaries()
    plain_ms = {k: float(np.median(timed(stream, f, args.warmup, args.reps))) for k, f in calls.items()}
    up0, down0 = e.atmosphere_fluxes(mu, wt)
    out["boundaries"] = {"emissivity_table": eps_table, "t_top_k": 2.725, "n_mu": 3, "plain_ms_median": plain_ms,
                         "plain_olr_w_m2": float(up0[-1]), "plain_surface_net_w_m2": float(up0[0] - down0[0]),
                         "runs": []}
    try:
        for reflection in ("lambertian", "specular"):
            e.set_flux_boundaries(eps_table, reflection, 2.725)
            run = {"reflection": reflection}
            for k, f in calls.items():
                ms = timed(stream, f, args.warmup, args.reps)
                med = float(np.median(ms))
                run[k] = {"ms_median": med, "ms_p10_p90": [float(np.percentile(ms, 10)), float(np.percentile(ms, 90))],
                          "reps": args.reps, "ratio_to_plain_call": med / plain_ms[k]}
            up, down = e.atmosphere_fluxes(mu, wt)
            run.update(olr_w_m2=float(up[-1]), surface_net_w_m2=float(up[0] - down[0]), top_down_w_m2=float(down[-1]))
            out["boundaries"]["runs"].append(run)
    finally:
        e.set_flux_boundaries()
    out["solar"] = solar_section(e, stream, args, w, mu, wt, calls, eps_table)
    out["continuum"] = continuum_section(e, stream, w, column, mu, wt, rrtmg, peaks["copy_bytes_per_s"])
    out["kernels"] = kernels_section(e, stream, args, w, column, mu, wt, rrtmg)
    e.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
