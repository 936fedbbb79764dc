"""The bench.py JSON contract on CPU: the reference arm (the oracle port on the host cores) prints ONE line with the
keys the driver reads, on the same metric / unit / config as the GPU arm."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "line-gridpoint evals/s" and d["unit"] == "pairs/s"
    assert d["higher_is_better"] is True and d["value"] > 1e6 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "cfg2" in d["config"]["workload"]


def test_gpu_arm_declares_the_same_metric():
    import bench
    assert bench.METRIC == "line-gridpoint evals/s" and bench.UNIT == "pairs/s"
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert bench.METRIC.split()[0] in base["metric"]


def test_real_reference_timing_fixture_describes_cfg1():
    """tests/golden/reference_cfg1_timing.json (the real, unmodified reference timed on cfg1 in the build container,
    scripts/time_reference_cfg1.py) is on the workload bench.py's cfg1 object runs: same lines, same accumulate count, and the
    timed run itself agreed with the oracle."""
    import numpy as np
    from oracle import physics as ph
    from pyrad_b200 import workloads
    d = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_cfg1_timing.json")))
    w = workloads.cfg1()
    n = ph.grid_len(w["range_min"], w["range_max"], w["res"])
    ln = w["per_group_lines"][0]
    lo, hi = ph.effective_range(w["range_min"], w["range_max"], w["cutoff"])
    nu = ln["nu"][(ln["nu"] > lo) & (ln["nu"] < hi)]
    assert d["pairs"] == ph.pair_count(ph.line_index(nu, w["range_min"], w["res"]), n, ph.window_len(w["cutoff"], w["res"]))
    assert d["cores"] == 1 and d["get_transmittance_s"] > 1.0 and d["max_abs_T_diff_oracle_vs_reference"] <= 1e-13


def test_dump_outputs_writes_float_arrays_and_a_fixed_sample_above_64_mb(tmp_path):
    """bench.dump_outputs: small outputs are written whole; outputs above the 64 MB budget are cut to one seeded sample of
    positions, the same for every array and every run, and stay within the budget with their .npy headers."""
    import numpy as np
    import bench
    small = {"radiance": np.linspace(0, 1, 1000, dtype=np.float32), "transmittance": np.arange(7, dtype=np.float64)}
    bench.dump_outputs(str(tmp_path / "small"), small)
    for name, a in small.items():
        got = np.load(str(tmp_path / "small" / (name + ".npy")))
        assert got.dtype == a.dtype and np.array_equal(got, a)
    n = 10_000_000                                       # 2 x 40 MB of float32
    big = {"radiance": np.arange(n, dtype=np.float32), "transmittance": -np.arange(n, dtype=np.float32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), big)
    sizes = [os.path.getsize(str(tmp_path / "a" / f)) for f in ("radiance.npy", "transmittance.npy")]
    assert sum(sizes) <= bench.DUMP_MAX_BYTES
    rad, tr = (np.load(str(tmp_path / "a" / f)) for f in ("radiance.npy", "transmittance.npy"))
    assert rad.dtype == np.float32 and rad.size > n // 2 and np.all(np.diff(rad) > 0)      # sorted positions, no repeats
    assert np.array_equal(tr, -rad)                                                        # one sample for both arrays
    assert np.array_equal(np.load(str(tmp_path / "b" / "radiance.npy")), rad)              # and for every run


def test_step_outputs_leave_out_only_the_radiance_at_zero_wavenumber():
    """The radiance is NaN at 0 cm-1 by design (Planck's 0/0, as the reference): the dump drops that one point of the
    radiance and nothing else, whatever the values, so a NaN anywhere else still reaches the dumped arrays; the
    transmittance is kept whole."""
    import numpy as np
    import bench

    class FakeEngine:
        def atmosphere_read_f32(self, rad, tr):
            rad[:] = np.arange(rad.size, dtype=np.float32)
            rad[0] = rad[5] = np.nan
            tr[:] = np.arange(tr.size, dtype=np.float32) / 10

    out = bench.step_outputs(FakeEngine(), 10, 1, None, 0.0)
    assert out["radiance"].size == 9 and out["radiance"][1] == 2.0
    assert np.isnan(out["radiance"][4]) and np.isfinite(np.delete(out["radiance"], 4)).all()
    assert np.array_equal(out["transmittance"], np.arange(10, dtype=np.float32) / 10)
    out = bench.step_outputs(FakeEngine(), 10, 1, None, 600.0)
    assert out["radiance"].size == out["transmittance"].size == 10 and np.isnan(out["radiance"][0])


@pytest.mark.gpu
def test_gpu_arm_dumps_the_step_result(tmp_path):
    """bench.py --dump-outputs writes what the timed step returns: equal, bit for bit, to the same step run again here on
    a fresh engine (same arguments, same outputs), with nothing non-finite beyond the radiance's 0 cm-1 point."""
    import numpy as np
    from pyrad_b200 import engine as eng
    from pyrad_b200 import workloads
    d = str(tmp_path / "dump")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-atmosphere",
                          "--no-cpu", "--no-farfield", "--dump-outputs", d], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    assert sorted(os.listdir(d)) == ["radiance.npy", "transmittance.npy"]
    rad_d, tr_d = (np.load(os.path.join(d, n + ".npy")) for n in ("radiance", "transmittance"))
    w = workloads.cfg2_shard(0, 1)
    sp, T, P = w["species"], w["T"], w["P"]
    with eng.Engine(0) as e:
        e.upload_lines(w["lines"], n_groups=len(sp))
        e.set_grid(w["range_min"], w["res"], w["n_total"], w["i_begin"], w["i_end"])
        e.atmosphere([w["depth_cm"]], [T], [P], [w["conc"]], [s.molmass for s in sp], [[s.q(T) for s in sp]],
                     [s.q296 for s in sp], [eng.window_len(w["cutoff"], w["res"])], w["t_surface"], w["range_max"])
        rad, tr = np.empty(e.n_chunk, dtype=np.float32), np.empty(e.n_chunk, dtype=np.float32)
        e.atmosphere_read_f32(rad, tr)
    assert rad_d.dtype == tr_d.dtype == np.float32 and tr_d.shape == (3_000_000,) and rad_d.shape == (3_000_000 - 1,)
    assert np.array_equal(tr_d.view(np.int32), tr.view(np.int32))
    assert np.isnan(rad[0]) and np.array_equal(rad_d.view(np.int32), rad[1:].view(np.int32))
    assert np.isfinite(rad_d).all() and np.isfinite(tr_d).all() and 0 <= tr_d.min() <= tr_d.max() <= 1


def test_bench_rejects_zero_steps():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--steps" in out.stderr


def test_rank_affinity_helper_never_fails_and_never_widens():
    """bench.pin_rank_to_gpu_numa binds a rank to its GPU's CPUs when the box tells which those are; without nvidia-smi or
    sysfs (here) it reports why nothing changed and leaves the affinity alone."""
    import bench
    before = os.sched_getaffinity(0)
    msg = bench.pin_rank_to_gpu_numa(0)
    assert isinstance(msg, str) and msg
    assert os.sched_getaffinity(0) <= before
    os.sched_setaffinity(0, before)
