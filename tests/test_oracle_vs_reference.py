"""CPU tests: the oracle against the REAL reference executed live through oracle/ref_harness.py, from the sources
PYRAD_REFERENCE_DIR points to; skipped where they are absent.  Without them only part of this pin remains: the committed
golden vectors (tests/test_oracle.py) hold the oracle to the reference's outputs on fixed gas cells, xsc tables, the xsc
file utilities and known answers, but nothing stored covers what these tests check -- mergeArray on random ranges, the
layer mutation model, the text readers and random cells at dynamic and 0.002 base resolution."""
import numpy as np
import pytest

from oracle import physics as ph
from oracle import ref_harness as rh
from pyrad_b200 import synth

pytestmark = pytest.mark.skipif(not rh.available(), reason="reference sources not mounted")


def test_real_reference_loop_equals_oracle(tmp_path):
    wd = str(tmp_path)
    sp = synth.species("co2")
    lines = synth.make_lines(250, 595.2, 704.8, 1)
    rh.seed_workdir(wd)
    rh.write_params(wd, sp.global_iso, "co2", sp.mol_id, 626, 0.98, sp.q296, 1, sp.molmass)
    rh.write_q_table(wd, sp.global_iso, range(100, 400), [sp.q(t) for t in range(100, 400)])
    rh.write_line_segments(wd, sp.global_iso, sp.mol_id, 1, lines, 500, 800)
    ref = rh.load_reference(wd)
    C = ref.classes
    with rh.quiet():
        layer = C.Layer(10, 250, 500.0, 600, 700)
        mol = layer.addMolecule("co2", ppm=400)
        sig = C.getCrossSection(mol[0])
        tr = C.getTransmittance(layer)
        surf = ref.planck.planckWavenumber(layer.xAxis, 288)
        rad = layer.transmission(surf)
    lo, hi = ph.effective_range(600, 700, ph.layer_cutoff(500.0))
    m = (lines["nu"] > lo) & (lines["nu"] < hi)
    sub = {k: v[m] for k, v in lines.items()}
    assert np.array_equal([l.wavenumber for l in mol[0]], sub["nu"])
    args = (sub, 250, 500.0, 400e-6, sp.molmass, sp.q(250), sp.q296, 600, 700, 0.01, ph.layer_cutoff(500.0))
    o = ph.cross_section(*args)
    np.testing.assert_allclose(o, sig, rtol=1e-13, atol=0)
    pts = np.array([0, 1, 5, 100, 5000, 9998, 9999])
    np.testing.assert_allclose(ph.cross_section_at(pts, *args), sig[pts], rtol=1e-13)
    t = ph.transmittance(ph.abs_coef(o, 400e-6, 500.0, 250), 10)
    np.testing.assert_allclose(t, tr, rtol=1e-13)
    xa = ph.x_axis(600, 700, .01)
    np.testing.assert_array_equal(xa, layer.xAxis)
    np.testing.assert_allclose(ph.transmission(t, ph.planck_wavenumber(xa, 288), ph.planck_wavenumber(xa, 250)), rad, rtol=1e-13)
    # accumulation count of the reference loop == the metric's pair definition
    n = ph.grid_len(600, 700, .01)
    W = ph.window_len(ph.layer_cutoff(500.0), .01)
    idx = ph.line_index(sub["nu"], 600, .01)
    brute = sum(sum(1 for d in range(-(W - 2), W - 1) if 0 <= i + d <= n - 1) for i in idx)
    assert ph.pair_count(idx, n, W) == brute


def test_real_reference_merge_array_random_ranges(tmp_path):
    """mergeArray of the real reference against the oracle's restatement on random layer / table ranges: the same array
    or the same exception (its `.index` lookups raise ValueError off the 0.01 lattice, its copy loop IndexError)."""
    ref = rh.load_reference(str(tmp_path))
    rng = np.random.default_rng(23)
    same = raised = 0
    for _ in range(250):
        a = round(float(rng.uniform(500.0, 600.0)), int(rng.integers(0, 4)))
        b = a + round(float(rng.uniform(0.5, 30.0)), int(rng.integers(0, 3)))
        new_x = np.linspace(a, b, int((b - a) / .01))
        lo = round(float(rng.uniform(a - 25.0, b + 8.0)), int(rng.integers(0, 4)))
        hi = lo + round(float(rng.uniform(0.2, 50.0)), int(rng.integers(0, 3)))
        old_x = np.arange(lo, hi, .01)
        if len(new_x) < 2 or len(old_x) < 2:
            continue
        old_y = rng.uniform(1, 2, old_x.size)
        try:
            want = ref.classes.mergeArray(new_x, old_x, old_y)
        except (ValueError, IndexError) as err:
            with pytest.raises(type(err)):
                ph.merge_array(new_x, old_x, old_y)
            raised += 1
            continue
        got = ph.merge_array(new_x, old_x, old_y)
        assert np.array_equal(got, want)
        same += 1
    assert same > 40 and raised > 5


@pytest.mark.parametrize("seed", range(16))
def test_real_reference_random_cells_equal_oracle(tmp_path, seed):
    """Random small gas cells through the REAL reference (its scalar loop: a second or two each) against the oracle:
    pressure decides the line-shape regime and the window, temperature the Q lookup, two species, base resolution
    0.01 or (overridden, SURVEY 8(a) a11) 0.002."""
    rng = np.random.default_rng(900 + seed)
    wd = str(tmp_path)
    P = float(np.exp(rng.uniform(np.log(0.05), np.log(2000.0))))
    T = int(rng.integers(190, 320))
    base = float(rng.choice([0.01, 0.002]))
    dynamic = bool(base == 0.01 and rng.random() < 0.5)                  # pyradClasses.py:659-662: coarser grid above 10 atm
    if dynamic:
        P = float(np.exp(rng.uniform(np.log(10200.0), np.log(30000.0))))
    rmin = float(rng.choice([600.0, 1000.0, 2349.0]))
    rmax = rmin + float(rng.uniform(2.0, 12.0)) * (base / 0.01) * (10.0 if dynamic else 1.0)
    names = ["co2", "h2o"][: int(rng.integers(1, 3))]
    conc = [400e-6, 0.01][: len(names)]
    cutoff = ph.layer_cutoff(P)
    rh.seed_workdir(wd)
    per = []
    for g, nme in enumerate(names):
        sp = synth.species(nme)
        n_ln = int(rng.integers(20, 120))
        ln = synth.make_lines(n_ln, max(rmin - cutoff - 1.0, 0.0), rmax + cutoff + 1.0, 40 + 7 * seed + g)
        per.append((sp, ln))
        rh.write_params(wd, sp.global_iso, nme, sp.mol_id, 1, 0.99, sp.q296, 1, sp.molmass)
        rh.write_q_table(wd, sp.global_iso, range(100, 400), [sp.q(t) for t in range(100, 400)])
        rh.write_line_segments(wd, sp.global_iso, sp.mol_id, 1, ln, int(max(rmin - cutoff - 1.0, 0.0) / 100) * 100,
                               rmax + cutoff + 102)
    ref = rh.load_reference(wd)
    ref.set_base_resolution(base)
    C = ref.classes
    with rh.quiet():
        layer = C.Layer(25.0, T, P, rmin, rmax, dynamicResolution=dynamic)
        mols = [layer.addMolecule(nme, concentration=c) for nme, c in zip(names, conc)]
        sig = [np.asarray(C.getCrossSection(m[0])) for m in mols]
        k = np.asarray(C.getAbsCoef(layer))
        tr = np.asarray(C.getTransmittance(layer))
    res = ph.layer_resolution(P, base, dynamic)
    assert layer.resolution == res and (not dynamic or res > base)
    lo, hi = ph.effective_range(rmin, rmax, cutoff)
    k_or = 0
    for (sp, ln), c, s_ref, m in zip(per, conc, sig, mols):
        keep = (ln["nu"] > lo) & (ln["nu"] < hi)
        sub = {kk: v[keep] for kk, v in ln.items()}
        assert np.array_equal([l.wavenumber for l in m[0]], sub["nu"])
        o = ph.cross_section(sub, T, P, c, sp.molmass, sp.q(T), sp.q296, rmin, rmax, res, cutoff)
        if res != base:
            o = ph.interp_to_base(o, rmin, rmax, res, base)
        np.testing.assert_allclose(o, s_ref, rtol=1e-12, atol=0)
        k_or = k_or + ph.abs_coef(o, c, P, T)
    np.testing.assert_allclose(k_or, k, rtol=1e-12, atol=0)
    np.testing.assert_allclose(ph.transmittance(k_or, 25.0), tr, rtol=1e-12, atol=0)


@pytest.mark.parametrize("seed", range(8))
def test_real_reference_layer_mutations_equal_the_state_model(tmp_path, seed):
    """changeTemperature / changePressure / changeDepth / setPPM / changeRange on a REAL reference layer, k and T after
    every step against tests.helpers.LayerModel -- the model the GPU sweep then holds the host mirror to."""
    from tests import helpers as H
    case = H.random_layer_case(seed)
    wd = str(tmp_path)
    rh.seed_workdir(wd)
    H.seed_layer_case(wd, case, rh)
    ref = rh.load_reference(wd)
    model = H.LayerModel(case["species"], case["lines"], case["conc"], case["depth"], case["T"], case["P"], case["rmin"],
                         case["rmax"])

    def check(layer, model, tag):
        with rh.quiet():
            k = np.asarray(ref.classes.getAbsCoef(layer))
            t = np.asarray(ref.classes.getTransmittance(layer))
        assert layer.resolution == model.res and layer.distanceFromCenter == model.cutoff, tag
        np.testing.assert_allclose(k, model.abs_coef(), rtol=1e-12, atol=0, err_msg=str(tag))
        np.testing.assert_allclose(t, model.transmittance(), rtol=1e-12, atol=0, err_msg=str(tag))
        # what the menus derive from it (pyradClasses.py:26-29, 73-88) and the line survey made at load time
        with rh.quiet():
            tau, ab, em = (np.asarray(f(layer)) for f in (ref.classes.getOpticalDepth, ref.classes.getAbsorbance,
                                                           ref.classes.getEmissivity))
            surv = np.asarray(layer.lineSurvey)
            total = ref.classes.integrateSpectrum(em, res=.01)
        tm = model.transmittance()
        np.testing.assert_allclose(tau, ph.optical_depth(tm), rtol=1e-9, atol=1e-15, err_msg=str(tag))
        np.testing.assert_allclose(ab, ph.absorbance(tm), rtol=1e-9, atol=1e-15, err_msg=str(tag))
        np.testing.assert_allclose(em, ph.emissivity(tm), rtol=1e-9, atol=1e-15, err_msg=str(tag))
        assert np.array_equal(surv, model.line_survey()), tag
        assert total == pytest.approx(ph.integrate_spectrum(ph.emissivity(tm), res=.01), rel=1e-9)

    with rh.quiet():
        H.drive_layer_case(ref.classes, case, model, check)


def test_real_reference_readers_on_random_text(tmp_path):
    """readHitranOnlineFile and returnXscFileContents of the real reference on random well-formed files (the cell formats,
    row orders, repeated wavenumbers, CRLF, range bounds of tests/test_gpu_fuzz.py's text sweeps; the reference crashes
    on a comment row below the header and on a malformed xsc row, so those stay out here) against the oracle's readers,
    which the device parsers are then held to on the GPU."""
    import os
    from tests.test_gpu_fuzz import make_csv_case
    ref = rh.load_reference(str(tmp_path))
    rng = np.random.default_rng(5)
    checked = 0
    for seed in range(60):
        text, data_rows, lo, hi = make_csv_case(seed)
        if not data_rows:
            continue
        eol = "\r\n" if text.startswith("# header\r") else "\n"
        path = os.path.join(str(tmp_path), "seg_%d.pyr" % seed)
        with open(path, "w", newline="") as f:
            f.write("# header" + eol + eol.join(r.rstrip("\r") for r in data_rows) + eol)
        want = ref.utils.readHitranOnlineFile(path, lo, hi)
        got = ph.read_hitran_online_rows(data_rows, lo, hi)
        assert list(want.keys()) == list(got["nu"])
        for j, (nu, c) in enumerate(want.items()):
            assert (c["intensity"], c["einsteinA"], c["lowerEnergy"], c["airHalfWidth"], c["selfHalfWidth"], c["tempExponent"],
                    c["pressureShift"]) == (got["sw"][j], got["a"][j], got["elower"][j], got["gamma_air"][j],
                                            got["gamma_self"][j], got["n_air"][j], got["delta_air"][j])
        checked += 1
    assert checked > 40
    for seed in range(20):
        n = int(rng.integers(1, 400))
        x = 700.0 + 0.02 * np.arange(n)
        y = 10.0 ** rng.uniform(-24, -17, n)
        fm = [repr, lambda v: "%.6f" % v, lambda v: "%.4E" % v, lambda v: "%+.5E" % v]
        rows = [" " * int(rng.integers(0, 3)) + fm[int(rng.integers(0, 4))](float(a)) + " " * int(rng.integers(1, 8)) +
                fm[int(rng.integers(0, 4))](float(b)) + " " * int(rng.integers(0, 3)) for a, b in zip(x, y)]
        path = os.path.join(str(tmp_path), "xsc_%d.txt" % seed)
        with open(path, "w") as f:
            f.write("# header\n" + "\n".join(rows) + "\n")
        with rh.quiet():
            want = ref.utils.returnXscFileContents(path)
        wn, xs = ph.read_xsc_rows(rows)
        assert want["wavenumber"] == list(wn) and want["intensity"] == list(xs)
