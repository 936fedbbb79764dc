"""Generate tests/golden/*.npz by running the REAL, UNMODIFIED reference (bschrag620/PyRad mounted at
/root/reference) through oracle/ref_harness.py on seeded synthetic HITRAN-format data.

Run in the build container only:   python tests/golden/make_golden.py
The reference is Python and cannot travel to the GPU box, so these vectors are the pin that does:
the oracle is checked against them on CPU, the CUDA engine on the GPU.  Every file stores the inputs
(line columns, species constants, layer scalars) next to the reference's outputs, so no test needs
/root/reference at run time.
"""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import ref_harness as rh          # noqa: E402
from pyrad_b200 import synth                  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
LOCAL_ISO = 1


def seed_species(wd, sp, lines, seg_lo, seg_hi):
    rh.write_params(wd, sp.global_iso, sp.name, sp.mol_id, 1, 0.99, sp.q296, 1, sp.molmass)
    rh.write_q_table(wd, sp.global_iso, range(100, 501), [sp.q(t) for t in range(100, 501)])
    rh.write_line_segments(wd, sp.global_iso, sp.mol_id, LOCAL_ISO, lines, seg_lo, seg_hi)


def pack_lines(prefix, lines):
    return {"%s_%s" % (prefix, k): np.asarray(v) for k, v in lines.items()}


def case_gas_cell(name, species_names, conc, n_lines, rmin, rmax, T, P, depth, seed, base=None, dynamic=True,
                  surface_T=288):
    wd = tempfile.mkdtemp(prefix="pyrad_golden_")
    sps = [synth.species(s) for s in species_names]
    rh.seed_workdir(wd)
    cutoff = P / 1013.25 * 5
    lo, hi = max(rmin - cutoff, 0.0), rmax + cutoff
    all_lines = []
    for g, sp in enumerate(sps):
        ln = synth.make_lines(n_lines, max(lo - 1.0, 0.0), hi + 1.0, seed + 17 * g)   # some lines fall outside the kept range
        seed_species(wd, sp, ln, int(max(lo - 1.0, 0.0) / 100) * 100, hi + 101.0)
        all_lines.append(ln)
    ref = rh.load_reference(wd)
    if base is not None:
        ref.set_base_resolution(base)
    C = ref.classes
    out = {"species": np.array(species_names), "conc": np.array(conc, dtype=np.float64),
           "molmass": np.array([s.molmass for s in sps]), "q296": np.array([s.q296 for s in sps]),
           "qT": np.array([s.q(T) for s in sps]),
           "T": T, "P": P, "depth": depth, "range_min": rmin, "range_max": rmax, "surface_T": surface_T,
           "base": ref.utils.BASE_RESOLUTION, "dynamic": dynamic}
    with rh.quiet():
        layer = C.Layer(depth, T, P, rmin, rmax, dynamicResolution=dynamic)
        mols = []
        for sp, c in zip(sps, conc):
            mols.append(layer.addMolecule(sp.name, concentration=c))
        out["res"] = layer.resolution
        out["cutoff"] = layer.distanceFromCenter
        out["xaxis"] = np.asarray(layer.xAxis)
        for g, m in enumerate(mols):
            iso = m[0]
            out["kept_nu_%d" % g] = np.array([l.wavenumber for l in iso])
            out["sigma_%d" % g] = np.asarray(C.getCrossSection(iso))
            out["abscoef_%d" % g] = np.asarray(C.getAbsCoef(m))
        out["layer_abscoef"] = np.asarray(C.getAbsCoef(layer))
        out["layer_transmittance"] = np.asarray(C.getTransmittance(layer))
        surf = ref.planck.planckWavenumber(layer.xAxis, surface_T)
        out["surface"] = np.asarray(surf)
        out["layer_transmission"] = np.asarray(layer.transmission(surf))
        out["layer_planck"] = np.asarray(layer.planck(layer.T))
        # section 8(f) rows: line survey, derived spectra, integrated radiance
        for g, m in enumerate(mols):
            out["survey_%d" % g] = np.asarray(m[0].createLineSurvey())
        out["layer_survey"] = np.asarray(layer.lineSurvey)
        with np.errstate(all="ignore"):
            out["layer_optical_depth"] = np.asarray(C.getOpticalDepth(layer))
            out["layer_absorbance"] = np.asarray(C.getAbsorbance(layer))
            out["layer_emissivity"] = np.asarray(C.getEmissivity(layer))
        out["integrated_transmission"] = float(C.integrateSpectrum(out["layer_transmission"], res=ref.utils.BASE_RESOLUTION))
        out["integrated_surface"] = float(C.integrateSpectrum(out["surface"], res=ref.utils.BASE_RESOLUTION))
    for g, ln in enumerate(all_lines):
        out.update(pack_lines("lines%d" % g, ln))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "N=%d res=%g W-cutoff=%g kept=%s" % (len(out["layer_abscoef"]), out["res"], out["cutoff"],
                                                    [len(out["kept_nu_%d" % g]) for g in range(len(sps))]))


def case_xsc(name, file_res, rmin_f, rmax_f, layer_rmin, layer_rmax, seed):
    """xsc molecule next to a line-by-line molecule (cfg3 in miniature).  The xsc branch overwrites the layer's
    T and P with the file's (pyradClasses.py:488-491)."""
    wd = tempfile.mkdtemp(prefix="pyrad_golden_")
    rh.seed_workdir(wd)
    sp = synth.species("co2")
    T_file, torr = 296, 760.0
    P_file = torr / 0.75006
    cutoff = P_file / 1013.25 * 5
    ln = synth.make_lines(300, max(layer_rmin - cutoff, 0), layer_rmax + cutoff, seed)
    seed_species(wd, sp, ln, int(max(layer_rmin - cutoff, 0) / 100) * 100, layer_rmax + cutoff + 101)
    fx, fy = synth.make_xsc_table(rmin_f, rmax_f, file_res, seed + 1)
    fname = rh.write_xsc_file(wd, "CFC11", float(T_file), torr, rmin_f, rmax_f, file_res, fx, fy)
    ref = rh.load_reference(wd)
    C = ref.classes
    out = {"file_x": fx, "file_y": fy, "file_res": file_res, "file_rmin": rmin_f, "file_rmax": rmax_f,
           "layer_rmin": layer_rmin, "layer_rmax": layer_rmax, "molmass": sp.molmass, "q296": sp.q296,
           "conc_xsc": 250e-12, "conc_co2": 400e-6, "depth": 100.0}
    with rh.quiet():
        layer = C.Layer(100.0, 250, 500.0, layer_rmin, layer_rmax)
        xm = layer.addMolecule({"CFC11": fname}, concentration=250e-12)
        out["T_after"] = layer.T
        out["P_after"] = layer.P
        m = layer.addMolecule("co2", concentration=400e-6)
        out["qT"] = sp.q(layer.T)
        out["xaxis"] = np.asarray(layer.xAxis)
        out["xsc_sigma"] = np.asarray(C.getCrossSection(xm), dtype=np.float64)
        out["co2_sigma"] = np.asarray(C.getCrossSection(m[0]))
        out["layer_abscoef"] = np.asarray(C.getAbsCoef(layer))
        out["layer_transmittance"] = np.asarray(C.getTransmittance(layer))
        out["res"] = layer.resolution
        out["cutoff"] = layer.distanceFromCenter
    out.update(pack_lines("lines0", ln))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "N=%d xsc nonzero=%d T,P after=%s,%s" % (len(out["xsc_sigma"]), int(np.count_nonzero(out["xsc_sigma"])),
                                                        out["T_after"], out["P_after"]))


def _folder_bytes(d):
    return {f: open(os.path.join(d, f), "rb").read() for f in sorted(os.listdir(d))}


def _pack_files(prefix, files):
    """{name: bytes} -> npz-friendly arrays: names (unicode), one uint8 blob, offsets."""
    names = sorted(files)
    blob = b"".join(files[n] for n in names)
    offs = np.cumsum([0] + [len(files[n]) for n in names])
    return {prefix + "_names": np.array(names), prefix + "_blob": np.frombuffer(blob, dtype=np.uint8),
            prefix + "_offsets": offs.astype(np.int64)}


def case_xsc_files(name):
    """SURVEY 8(f) row 4: the xsc FILE utilities run for real -- changeResXscFile (pyradUtilities.py:515-534: table ->
    np.interp onto arange(min, max, BASE_RESOLUTION) -> rewritten text file) and mergeXsc (:549-597: files of equal
    T and P summed onto the union range and rewritten).  Input and output folders are stored byte for byte."""
    wd = tempfile.mkdtemp(prefix="pyrad_golden_")
    rh.seed_workdir(wd)
    out = {}
    # (1) one coarse table per folder member: 0.05 and 0.03 cm-1 spacing, and one already at 0.01
    specs = [("CFC11", 296.0, 760.0, 830.0, 860.0, 0.05, 11), ("CFC11", 273.0, 7.5, 1050.0, 1062.0, 0.03, 12),
             ("CFC11", 253.0, 100.2, 810.0, 815.0, 0.01, 13)]
    for sp in specs:
        mol, T, torr, lo, hi, res, seed = sp
        fx, fy = synth.make_xsc_table(lo, hi, res, seed)
        rh.write_xsc_file(wd, mol, T, torr, lo, hi, res, fx, fy)
    d = os.path.join(wd, "data", "xsc", "CFC11")
    out.update(_pack_files("res_in", _folder_bytes(d)))
    ref = rh.load_reference(wd)
    with rh.quiet():
        for f in sorted(os.listdir(d)):
            ref.utils.changeResXscFile(os.path.join(d, f))
    out.update(_pack_files("res_out", _folder_bytes(d)))
    # (2) merge: folder of pyrad-adjusted files (the header glued to the first row, as writeXscFile leaves it) --
    # two (T, P) groups: three disjoint/abutting ranges at 296 K / 760 Torr, two at 250 K / 100 Torr
    d2 = os.path.join(wd, "data", "xsc", "HCFC22")
    os.makedirs(d2)
    groups = [(296.0, 760.0, [(800.0, 810.0, 21), (820.0, 835.0, 22), (835.0, 840.0, 23)]),
              (250.0, 100.0, [(1100.0, 1104.0, 24), (1090.0, 1095.0, 25)])]
    with rh.quiet():
        for T, torr, parts in groups:
            for lo, hi, seed in parts:
                x = np.arange(lo, hi, ref.utils.BASE_RESOLUTION)
                _, y = synth.make_xsc_table(lo, hi, 0.01, seed)
                ref.utils.writeXscFile(x, y[: len(x)], lo, hi, T, torr, "HCFC22", d2, "N2", "07-19")
    out.update(_pack_files("merge_in", _folder_bytes(d2)))
    with rh.quiet():
        ref.utils.mergeXsc("HCFC22")
    out.update(_pack_files("merge_out", _folder_bytes(d2)))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, {k: (list(v) if k.endswith("_names") else v.shape) for k, v in out.items()})


def case_cfg3_mini(name):
    """BASELINE cfg3 in miniature, run by the real reference: line-by-line CO2 + H2O next to TWO xsc tables (CFC-11 at
    its native 0.01 cm-1, HCFC-22 at 0.05 cm-1 -> np.interp) on one 0.01 cm-1 grid.  Both tables are 296 K / 760 Torr
    files, so the layer ends up at their T and P (pyradClasses.py:488-491)."""
    wd = tempfile.mkdtemp(prefix="pyrad_golden_")
    rh.seed_workdir(wd)
    rmin, rmax, depth = 600.0, 700.0, 10.0
    T_file, torr = 296, 760.0
    cutoff = torr / 0.75006 / 1013.25 * 5
    lo, hi = max(rmin - cutoff, 0.0), rmax + cutoff
    names, conc = ["co2", "h2o"], [400e-6, 0.01]
    sps = [synth.species(s) for s in names]
    all_lines = []
    for g, sp in enumerate(sps):
        ln = synth.make_lines(1200, lo - 1.0, hi + 1.0, 808 + 17 * g)
        seed_species(wd, sp, ln, int((lo - 1.0) / 100) * 100, hi + 101.0)
        all_lines.append(ln)
    tables = [("CFC11", 0.01, 620.0, 650.0, 250e-12, 811), ("HCFC22", 0.05, 660.0, 690.0, 230e-12, 812)]
    out = {"species": np.array(names), "conc": np.array(conc), "molmass": np.array([s.molmass for s in sps]),
           "q296": np.array([s.q296 for s in sps]), "range_min": rmin, "range_max": rmax, "depth": depth,
           "xsc_names": np.array([t[0] for t in tables]), "xsc_res": np.array([t[1] for t in tables]),
           "xsc_rmin": np.array([t[2] for t in tables]), "xsc_rmax": np.array([t[3] for t in tables]),
           "xsc_conc": np.array([t[4] for t in tables]), "surface_T": 288}
    fnames = []
    for i, (mol, res, a, b, _, seed) in enumerate(tables):
        fx, fy = synth.make_xsc_table(a, b, res, seed)
        fnames.append(rh.write_xsc_file(wd, mol, float(T_file), torr, a, b, res, fx, fy))
        out["xsc_x_%d" % i], out["xsc_y_%d" % i] = fx, fy
    ref = rh.load_reference(wd)
    C = ref.classes
    with rh.quiet():
        layer = C.Layer(depth, 280, 900.0, rmin, rmax)
        xms = [layer.addMolecule({t[0]: f}, concentration=t[4]) for t, f in zip(tables, fnames)]
        mols = [layer.addMolecule(n, concentration=c) for n, c in zip(names, conc)]
        out["T_after"], out["P_after"] = layer.T, layer.P
        out["qT"] = np.array([s.q(layer.T) for s in sps])
        out["res"], out["cutoff"] = layer.resolution, layer.distanceFromCenter
        out["xaxis"] = np.asarray(layer.xAxis)
        for i, xm in enumerate(xms):
            out["xsc_sigma_%d" % i] = np.asarray(C.getCrossSection(xm), dtype=np.float64)
        for g, m in enumerate(mols):
            out["sigma_%d" % g] = np.asarray(C.getCrossSection(m[0]))
        out["layer_abscoef"] = np.asarray(C.getAbsCoef(layer))
        out["layer_transmittance"] = np.asarray(C.getTransmittance(layer))
        surf = ref.planck.planckWavenumber(layer.xAxis, 288)
        out["layer_transmission"] = np.asarray(layer.transmission(surf))
    for g, ln in enumerate(all_lines):
        out.update(pack_lines("lines%d" % g, ln))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "N=%d T,P after=%s,%s xsc nonzero=%s" % (len(out["layer_abscoef"]), out["T_after"], out["P_after"],
                                                         [int(np.count_nonzero(out["xsc_sigma_%d" % i])) for i in range(2)]))


def case_kat(name):
    """Known-answer values straight from the real physics modules (SURVEY.md section 8(c))."""
    wd = tempfile.mkdtemp(prefix="pyrad_golden_")
    ref = rh.load_reference(wd)
    I, L, Pk = ref.intensity, ref.lineshape, ref.planck
    m = 43.98983 / 1000 / 6.022140857E23
    g = L.gaussianHW(667.661, 250, m)
    l = L.lorentzHW(.07, .09, 500., 250, 4e-4, .7)
    l2 = L.lorentzHW(.07, .09, 10., 250, 4e-4, .7)
    x = np.array([0, .01, .1, 1])
    x2 = np.array([0, .001, .002, .01])
    out = {
        "c2": I.c2, "boltz": I.boltzmannFactors(100, 250), "stim": I.stimulatedEmissions(667.661, 250),
        "intensity": I.intensityFactor(3.0e-19, 667.661, 250, 100.0, 220.0, 286.09),
        "m": m, "gHW": g, "lHW": l, "lHW2": l2,
        "x": x, "x2": x2,
        "lorentz": L.lorentzLineShape(l, x), "voigt": L.pseudoVoigtShape(g, l, x), "gauss0": L.gaussianLineShape(g, 0),
        "gauss": L.gaussianLineShape(g, x2), "voigt2": L.pseudoVoigtShape(g, l2, x2),
        "planck": Pk.planckWavenumber(np.array([1., 667., 2000.]), 288),
    }
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, {k: (v if np.ndim(v) == 0 else "...") for k, v in out.items()})


def case_hitran_id_tables(name):
    """MOLECULE_ID and HITRAN_GLOBAL_ISO read from the reference source's dict literals (pyradClasses.py:951-1022)."""
    with open(os.path.join(OUT, name + ".json"), "w") as f:
        f.write(rh.id_tables_json(rh.reference_id_tables()))
    print(name, "written")


if __name__ == "__main__":
    if not rh.available():
        raise SystemExit("the reference is not mounted at %s" % rh.REFERENCE_DIR)
    if len(sys.argv) > 1:                                          # regenerate only the named late additions
        {"xsc_files": case_xsc_files, "cfg3_mini": case_cfg3_mini,
         "hitran_id_tables": case_hitran_id_tables}[sys.argv[1]](sys.argv[1])
        raise SystemExit(0)
    case_kat("kat")
    case_gas_cell("cell_co2_1atm", ["co2"], [400e-6], 1500, 600.0, 700.0, 296, 1013.0, 10.0, 101)
    case_gas_cell("cell_lowp", ["co2", "h2o"], [400e-6, 0.005], 900, 640.0, 690.0, 220, 5.0, 1000.0, 202)
    case_gas_cell("cell_tiny_window", ["co2"], [400e-6], 600, 660.0, 680.0, 200, 0.05, 1e5, 303)
    case_gas_cell("cell_fine_grid", ["h2o", "co2"], [0.01, 400e-6], 700, 1000.0, 1008.0, 280, 800.0, 50.0, 404,
                  base=0.001, dynamic=False)
    case_gas_cell("cell_highp_dynres", ["co2"], [0.02], 400, 600.0, 700.0, 300, 20000.0, 5.0, 505)
    case_xsc("xsc_native_res", 0.01, 830.0, 860.0, 800.0, 900.0, 606)
    case_xsc("xsc_coarse_res", 0.05, 830.0, 860.0, 800.0, 900.0, 707)
    case_xsc_files("xsc_files")
    case_cfg3_mini("cfg3_mini")
    case_hitran_id_tables("hitran_id_tables")
