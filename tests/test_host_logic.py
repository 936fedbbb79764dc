"""CPU tests of host-side logic that needs no device: numpy-compatible helpers, workloads, the mirror's
bookkeeping, bench plumbing."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import physics as ph
from pyrad_b200 import classes as C
from pyrad_b200 import engine as eng
from pyrad_b200 import synth
from pyrad_b200 import workloads

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_linspace_axis_reproduces_numpy_bitwise():
    for a, b, n in [(600.0, 700.0, 10000), (0.0, 3000.0, 3000000), (1000.0, 1008.0, 8000), (600.0, 600.1, 1),
                    (600.0, 600.1, 2)]:
        x0, dx, xl, n_ = eng.linspace_axis(a, b, n)
        ref = np.linspace(a, b, n, endpoint=True)
        mine = np.arange(n) * dx + x0
        mine[-1] = xl
        assert np.array_equal(mine, ref)


def test_window_and_grid_rules_follow_numpy():
    assert eng.window_len(5 * 1013 / 1013.25, .01) == 500
    assert eng.window_len(25, .001) == 25000
    assert eng.window_len(0.000246731, .01) == 1
    assert eng.grid_len(600.0, 607.77, 0.01) == int((607.77 - 600.0) / 0.01)
    assert eng.number_density_weight(4e-4, 1013.25, 296) == 4e-4 * 1013.25 / 1E4 / 1.38064852E-23 / 296


def test_workloads_are_seeded_sorted_and_shaped():
    w1, w2 = workloads.cfg1(2000), workloads.cfg1(2000)
    assert np.array_equal(w1["lines"]["nu"], w2["lines"]["nu"])
    assert np.all(np.diff(w1["lines"]["nu"]) > 0)
    w = workloads.cfg2(4000, 30.0)
    assert set(np.unique(w["lines"]["group"])) == {0, 1, 2, 3}
    assert np.all(np.diff(w["lines"]["nu"]) >= 0)
    a = workloads.atmosphere(n_layers=10, n_lines=1000, rmax=50.0)
    assert a["conc"].shape == (10, 4) and np.all(np.diff(a["P"]) < 0)
    assert np.all(a["T"] == np.round(a["T"]))                # integer K: the reference's Q lookup needs it
    s0, s1 = workloads.cfg2_shard(0, 2, 4000, 30.0), workloads.cfg2_shard(1, 2, 4000, 30.0)
    assert s0["n_total"] == s1["n_total"] == 60000 and s0["i_end"] == s1["i_begin"] == 30000
    # the margin lines of neighbouring shards are the same physical lines
    edge0 = s0["lines"]["nu"][s0["lines"]["nu"] > 30.0 - 5]
    edge1 = s1["lines"]["nu"][s1["lines"]["nu"] < 30.0 + s0["cutoff"]]
    both = np.intersect1d(edge0, edge1)
    assert both.size > 0 and np.all((both > 30.0 - s0["cutoff"]) & (both < 30.0 + s0["cutoff"]))


def test_us_standard_atmosphere_anchor_points():
    t, p = synth.us_standard_atmosphere(0.0)
    assert abs(t - 288.15) < 1e-9 and abs(p - 1013.25) < 1e-9
    t, p = synth.us_standard_atmosphere(11.0)
    assert abs(t - 216.65) < 1e-6 and abs(p - 226.32) < 0.05
    t, p = synth.us_standard_atmosphere(47.0)
    assert abs(t - 270.65) < 1e-6 and abs(p - 1.1091) < 0.002


def test_merge_plan_matches_oracle_merge_array():
    rng = np.random.default_rng(3)
    new_x = np.linspace(800.0, 900.0, 10000)
    for lo, hi in [(830.0, 860.0), (800.0, 900.0), (805.5, 806.5)]:
        old_x = np.arange(lo, hi, .01)
        old_y = rng.uniform(1, 2, old_x.size)
        ref = ph.merge_array(new_x, old_x, old_y)
        dst0, src0, count, out_len = C._merge_plan(new_x, old_x)
        assert out_len == len(ref)
        mine = np.zeros(out_len)
        mine[dst0:dst0 + count] = old_y[src0:src0 + count]
        assert np.array_equal(mine, ref)
    # new range inside the old one
    old_x = np.arange(700.0, 1000.0, .01)
    old_y = rng.uniform(1, 2, old_x.size)
    ref = ph.merge_array(new_x, old_x, old_y)
    dst0, src0, count, out_len = C._merge_plan(new_x, old_x)
    mine = np.zeros(out_len)
    mine[dst0:dst0 + count] = old_y[src0:src0 + count]
    assert np.array_equal(mine, ref)


def test_merge_plan_random_ranges_behave_like_the_oracle():
    """Random layer / table ranges (table inside, around, overlapping one end of, or away from the layer's range; edges
    on and off the 0.01 grid): the plan reproduces mergeArray's result or fails where it fails (its `.index` lookups
    raise ValueError when a rounded edge is not on the other axis)."""
    rng = np.random.default_rng(17)
    same, raised = 0, 0
    for _ in range(300):
        a = round(float(rng.uniform(500.0, 600.0)), int(rng.integers(0, 4)))
        b = a + round(float(rng.uniform(0.5, 40.0)), int(rng.integers(0, 3)))
        new_x = np.linspace(a, b, int((b - a) / .01))                         # Layer.xAxis, pyradClasses.py:659
        lo = round(float(rng.uniform(a - 30.0, b + 10.0)), int(rng.integers(0, 4)))
        hi = lo + round(float(rng.uniform(0.2, 60.0)), int(rng.integers(0, 3)))
        old_x = np.arange(lo, hi, .01)
        if len(new_x) < 2 or len(old_x) < 2:
            continue
        old_y = rng.uniform(1, 2, old_x.size)
        try:
            ref = ph.merge_array(new_x, old_x, old_y)
        except (ValueError, IndexError) as err:
            with pytest.raises(type(err)):
                C._merge_plan(new_x, old_x)
            raised += 1
            continue
        dst0, src0, count, out_len = C._merge_plan(new_x, old_x)
        assert out_len == len(ref)
        mine = np.zeros(max(out_len, dst0 + count))
        mine[dst0:dst0 + count] = old_y[src0:src0 + count]
        assert np.array_equal(mine[:out_len], ref)
        same += 1
    assert same > 50 and raised > 5


def test_unit_conversions_and_concentration_setters():
    assert C.convertLength(2, "m") == 200 and C.convertPressure(1, "atm") == 1013.25
    assert C.convertRange(10, "um") == 1000 and C.convertTemperature(27, "C") == 300
    layer = C.Layer(10, 296, 1013.25, 600, 700)
    assert layer.distanceFromCenter == 5.0 and layer.resolution == .01
    assert len(layer.xAxis) == 10000 and layer.xAxis[1] - layer.xAxis[0] != .01      # linspace spacing, not res
    layer.changePressure(500.0)
    assert layer.distanceFromCenter == 500.0 / 1013.25 * 5
    assert layer.effectiveRangeMax == 705.0                                         # quirk: not updated


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "line-gridpoint evals/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0


def test_xsc_file_name_parser_matches_the_oracle():
    """Host logic of the xsc file utilities (no GPU): the product's parseXscFileName against the oracle's restatement
    of pyradUtilities.py:611-641 and against names the real reference wrote (tests/golden/xsc_files.npz)."""
    from oracle import physics as ph
    from pyrad_b200 import xsc_files as xf
    from tests import golden_util as G
    g = G.load("xsc_files")
    names = [str(n) for p in ("res_in", "res_out", "merge_in", "merge_out") for n in g[p + "_names"]]
    names.append("CFC-11_278.1K-760.3Torr_810.0-880.0_0.03_00_00.txt")     # no broadener field
    for n in names:
        got, want = xf.parseXscFileName(n), ph.parse_xsc_file_name(n)
        for k, v in want.items():
            assert got[k] == v, (n, k)
        assert got["LONG_FILENAME"] == n and got["SHORT_FILENAME"] + ".txt" == n


def test_hitran_id_tables_equal_the_reference_tables():
    """MOLECULE_ID and HITRAN_GLOBAL_ISO (pyradClasses.py:951-1022) carried in full: all 49 molecules and every
    isotopologue row, pinned by count and spot values, equal to tests/golden/hitran_id_tables.json on every run, and
    equal to the reference source's dict literals whenever the sources are present.  The committed JSON was written
    from pyrad_b200/hitran_tables.py (the tables this test holds equal to the reference source); make_golden.py
    hitran_id_tables rewrites it from the source itself."""
    from oracle import ref_harness as rh
    from pyrad_b200 import classes as C
    assert len(C.MOLECULE_ID) == 49 and sorted(C.MOLECULE_ID.values()) == list(range(1, 50))
    assert set(C.HITRAN_GLOBAL_ISO) == set(range(1, 50))
    assert sum(len(v) for v in C.HITRAN_GLOBAL_ISO.values()) == 126
    assert C.MOLECULE_ID["so2"] == 9 and C.MOLECULE_ID["nh3"] == 11 and C.MOLECULE_ID["cocl2"] == 49
    assert C.getGlobalIsotope(C.MOLECULE_ID["so2"], 2) == [42, 43]
    assert C.getGlobalIsotope(2, 12)[-1] == 122 and C.getGlobalIsotope(16, 2) == [19, 11]      # the reference's rows, sic
    with open(os.path.join(ROOT, "tests", "golden", "hitran_id_tables.json")) as f:
        g = json.load(f)
    assert g["MOLECULE_ID"] == C.MOLECULE_ID
    assert {int(m): {int(i): gid for i, gid in row.items()} for m, row in g["HITRAN_GLOBAL_ISO"].items()} == C.HITRAN_GLOBAL_ISO
    ref = rh.reference_id_tables()
    if ref is not None:
        assert ref["HITRAN_GLOBAL_ISO"] == C.HITRAN_GLOBAL_ISO
        assert ref["MOLECULE_ID"] == C.MOLECULE_ID


def test_reference_id_table_reader_and_golden_writer(tmp_path, monkeypatch):
    """The reader make_golden.py and the test above use on pyradClasses.py (dict literals found by brace matching,
    nested rows included) and the JSON layout of tests/golden/hitran_id_tables.json, on a stand-in source file."""
    from oracle import ref_harness as rh
    from pyrad_b200 import classes as C
    monkeypatch.setattr(rh, "REFERENCE_DIR", str(tmp_path))
    assert rh.reference_id_tables() is None
    with open(str(tmp_path / "pyradClasses.py"), "w") as f:
        f.write("import numpy as np\nx = {'a': {1: 2}}\nHITRAN_GLOBAL_ISO = %r\n\ndef f():\n    return {}\n\nMOLECULE_ID = %r\n"
                % (C.HITRAN_GLOBAL_ISO, C.MOLECULE_ID))
    tables = rh.reference_id_tables()
    assert tables == {"MOLECULE_ID": C.MOLECULE_ID, "HITRAN_GLOBAL_ISO": C.HITRAN_GLOBAL_ISO}
    with open(os.path.join(ROOT, "tests", "golden", "hitran_id_tables.json")) as f:
        assert rh.id_tables_json(tables) == f.read()


def test_isotope_lines_are_views_over_soa_columns(tmp_path, monkeypatch):
    """Isotope keeps the list protocol of the reference (pyradClasses.py:350-359: a list of Line objects) without
    holding one Python object per transition: len / iteration / indexing / linelist() hand out views on demand."""
    from oracle import ref_harness as rh          # only its data-tree writer (test infrastructure)
    root = str(tmp_path)
    sp = synth.species("co2")
    rh.write_params(root, sp.global_iso, sp.name, sp.mol_id, 1, 0.99, sp.q296, 1, sp.molmass)
    monkeypatch.setattr(C, "DATA_ROOT", root)
    monkeypatch.setattr(C.Layer, "hasAtmosphere", False)
    layer = C.Layer(10.0, 296, 1013.25, 600.0, 700.0)
    mol = C.Molecule("co2", layer, ppm=400)
    layer.append(mol)
    iso = mol[0]
    cols = synth.make_lines(1000, 590.0, 710.0, 5)
    iso.setLines(cols, {296: sp.q(296)})
    assert len(iso) == 1000 and bool(iso) and list.__len__(iso) == 0          # no per-line objects are stored
    first, last = iso[0], iso[-1]
    assert first.wavenumber == cols["nu"][0] and last.wavenumber == cols["nu"][-1]
    assert [ln.intensity for ln in iso[10:13]] == list(cols["sw"][10:13])
    assert sum(1 for _ in iso) == 1000 and len(iso.linelist()) == 1000 and len(C.totalLineList(layer)) == 1000
    ln = iso[5]
    assert ln.isotope is iso and ln.molecule is mol and ln.layer is layer
    assert ln.broadenedLine == cols["nu"][5] + cols["delta_air"][5] * layer.P / C.p0        # pyradClasses.py:252-254
    C.resetCrossSection(layer)                                                # does not walk the lines
    iso.clearLines()
    assert len(iso) == 0 and list(iso) == []
    np.testing.assert_raises(IndexError, lambda: iso[0])


def test_result_pool_without_a_device_returns_ordinary_arrays():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: covered by the gpu test")
    pool = eng.ResultPool()
    a = pool.array((3, 1 << 18))
    assert a.shape == (3, 1 << 18) and a.dtype == np.float64 and a.flags.owndata
