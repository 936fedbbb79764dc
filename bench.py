#!/usr/bin/env python
"""bench.py -- the headline measurement of pyrad-b200 (contract in the task statement / DESIGN.md).

Metric (BASELINE.json): line-gridpoint evals/s on the cfg2 gas cell (mixed H2O+CO2+CH4+O3, 0-3000 cm-1
at 0.001 cm-1, ~3M grid points, ~500k lines, Voigt, P = 1013.25 hPa => W = 5000), plus the 100-layer
atmosphere as a secondary object.  A "step" is one pass of the hot path over the cell: K1 prepass ->
K2 line sum -> K3 (exp(-k u), Planck, transmission).  With N ranks the spectrum is N consecutive
cfg2-sized wavenumber chunks (weak scaling, one chunk per GPU) and the finished transmittance spectra
are all-gathered once per step (the only collective).

  python bench.py [--gpus N --steps K --warmup W]          our arm (CUDA engine through the C ABI)
  python bench.py --impl reference [...]                   the reference's CPU path (oracle port) on the host cores
  python bench.py --dump-outputs DIR [...]                 also write the last timed step's spectra as DIR/<name>.npy
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "line-gridpoint evals/s"
UNIT = "pairs/s"
WORKLOAD = "cfg2: mixed H2O+CO2+CH4+O3 gas cell, 0-3000 cm-1 @ 0.001 cm-1 per GPU (3.0M points, ~500k lines, W=5000)"
SM_COUNT = 148
SM_MAX_MHZ_DEFAULT = 1965.0
DUMP_MAX_BYTES = 64_000_000
DUMP_SAMPLE_SEED = 20240601


def load_traffic(key):
    """DRAM bytes per launch of a kernel from the committed ncu --set full capture (profiles/traffic.json)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[key]
        return int(d["dram_bytes_read"]) + int(d["dram_bytes_write"])
    except Exception:
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            d = json.load(open(p))
            return d, "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "sm_max_mhz": SM_MAX_MHZ_DEFAULT}, "fallback"


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to fd 1
    when NCCL_DEBUG is set), so fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved
    descriptor."""
    sys.stdout.flush()
    keep = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(keep, "w")


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (recipe in B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.rows = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            c = [x.strip() for x in r.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
                pw.append(float(c[3]))
            except ValueError:
                continue
            for nme, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(np.max(mx)), "power_w_max": float(np.max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def pin_rank_to_gpu_numa(gpu_index):
    """Bind this rank's host threads to the CPUs local to its GPU (sysfs local_cpulist of the GPU's PCI device), before
    any pinned buffer is allocated: eight ranks streaming 56 MB per step through one socket's memory controllers is what
    the e2e number at N = 8 measured in round 1.  Returns a description for the JSON line; never fatal."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.count(":") == 2 and len(bus.split(":")[0]) == 8:
            bus = bus[4:]                                   # 00000000:1b:00.0 -> 0000:1b:00.0
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bus) as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "unchanged (GPU-local CPU list empty)"
        os.sched_setaffinity(0, cpus)
        return "GPU %d -> CPUs %s (%d)" % (gpu_index, spec, len(cpus))
    except Exception as exc:
        return "unchanged (%s)" % type(exc).__name__


def timed_runs(ext, run, reps, world, dist):
    """`reps` runs of `run`, each bracketed by a synchronise (+ barrier) and CUDA events on the launching stream."""
    import torch
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a.record(ext)
        run()
        b.record(ext)
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def max_over_ranks(values, world, dist):
    import torch
    t = torch.tensor([float(v) for v in values], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()]


def gather_parity(e, plan_chunks, nc, rank, world, dist):
    """Driver-visible multi-GPU evidence: the spectra the kernels stored into this rank's gather buffer over NVLink
    (peer stores + flag barrier) against a separate NCCL all-gather of every rank's local result, bit for bit."""
    import torch
    from pyrad_b200 import distributed as pd
    rad_g, tr_g = pd.gathered_spectra(e)
    rad_p, tr_p = e.atmosphere_result_dev()
    ld = rad_g.shape[1]
    ok = True
    for gathered, ptr in ((rad_g, rad_p), (tr_g, tr_p)):
        pad = torch.zeros(ld, dtype=torch.float32, device="cuda")
        pad[:nc] = pd.device_tensor(ptr, nc)
        ref = torch.empty(world * ld, dtype=torch.float32, device="cuda")
        dist.all_gather_into_tensor(ref, pad)
        ref = ref.view(world, ld)
        for r, (a, b) in enumerate(plan_chunks):
            # bit patterns, so that NaN (the reference's 0/0 at 0 cm-1) compares equal to itself
            ok = ok and bool(torch.equal(gathered[r, : b - a].view(torch.int32), ref[r, : b - a].view(torch.int32)))
    flag = torch.tensor([0 if ok else 1], dtype=torch.int32, device="cuda")
    dist.all_reduce(flag)
    return "bitwise" if int(flag.item()) == 0 else "MISMATCH on %d rank(s)" % int(flag.item())


def step_outputs(e, n_chunk, world, dist, range_min):
    """What a caller of the timed step receives from its last run: the float32 radiance and transmittance spectra
    (prb_atmosphere_read_f32), over the whole grid at N > 1 (every rank's chunk, in rank order).  Collective.

    The transmittance is whole.  The radiance leaves out a grid point at 0 cm-1: Planck's law as the reference
    evaluates it is 0/0 there, so the radiance is NaN by design (tests/test_gpu_parity.py holds the kernels to that)."""
    rad, tr = np.empty(n_chunk, dtype=np.float32), np.empty(n_chunk, dtype=np.float32)
    e.atmosphere_read_f32(rad, tr)
    out = {"radiance": rad, "transmittance": tr}
    if world > 1:
        import torch
        for name, mine in out.items():
            every = torch.empty(world * n_chunk, dtype=torch.float32, device="cuda")
            dist.all_gather_into_tensor(every, torch.from_numpy(mine).cuda())
            out[name] = every.cpu().numpy()
    if range_min == 0.0:
        out["radiance"] = out["radiance"][1:]
    return out


def dump_outputs(directory, arrays, max_bytes=DUMP_MAX_BYTES):
    """Write every array as directory/<name>.npy.  When they hold more than max_bytes together, each is cut to a sorted
    sample of its positions drawn with a fixed seed: the sample depends only on the array's length (arrays of one
    length share it), so runs with the same arguments write the same elements."""
    total = sum(a.nbytes for a in arrays.values())
    budget = max_bytes - 4096 * len(arrays)                   # room for the .npy headers
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        a = a.ravel()
        if total > budget:
            keep = a.size * budget // total
            a = a[np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(a.size, keep, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------- CPU side
def _oracle_window(args):
    """One bounded sample of the cfg2 workload on one core: the oracle's slice-add restatement of
    Isotope.createCrossSection on a `width` cm-1 sub-window of the cell, all four species."""
    lo, width, seed = args
    from oracle import physics as ph
    from pyrad_b200 import workloads
    w = workloads.gas_cell(["h2o", "co2", "ch4", "o3"], int(500_000 * (width + 10.0) / 3005.0), lo, lo + width, 0.001,
                           296, 1013.25, [0.01, 400e-6, 1.8e-6, 5e-8], 10.0, seed)
    t0 = time.perf_counter()
    pairs = 0
    n = ph.grid_len(w["range_min"], w["range_max"], w["res"])
    W = ph.window_len(w["cutoff"], w["res"])
    for g, sp in enumerate(w["species"]):
        ln = w["per_group_lines"][g]
        ph.cross_section(ln, w["T"], w["P"], w["conc"][g], sp.molmass, sp.q(w["T"]), sp.q296,
                         w["range_min"], w["range_max"], w["res"], w["cutoff"])
        pairs += ph.pair_count(ph.line_index(ln["nu"], w["range_min"], w["res"]), n, W)
    return pairs, time.perf_counter() - t0


def _literal_loop_rate():
    """The reference's OWN loop structure (pure-Python per-element scatter, pyradClasses.py:394-400) on a tiny
    sample -- context for how much faster the slice-add port is than the code it restates."""
    from oracle import physics as ph
    from pyrad_b200 import workloads
    w = workloads.gas_cell(["co2"], 60, 1000.0, 1010.0, 0.001, 296, 1013.25, [400e-6], 10.0, 4242)
    sp = w["species"][0]
    ln = w["per_group_lines"][0]
    t0 = time.perf_counter()
    ph.cross_section_scalar(ln, 296, 1013.25, 400e-6, sp.molmass, sp.q(296), sp.q296, 1000.0, 1010.0, 0.001, w["cutoff"])
    dt = time.perf_counter() - t0
    n = ph.grid_len(1000.0, 1010.0, 0.001)
    pairs = ph.pair_count(ph.line_index(ln["nu"], 1000.0, 0.001), n, ph.window_len(w["cutoff"], 0.001))
    return pairs / dt


def cpu_baseline_sample(budget_s=12.0):
    """Single-core oracle on successive 10 cm-1 windows of cfg2 until ~budget_s of CPU work is done."""
    pairs, secs, k = 0, 0.0, 0
    while secs < budget_s and k < 64:
        p, s = _oracle_window((1000.0 + 10.0 * k, 10.0, 777 + k))
        pairs += p
        secs += s
        k += 1
    lit = _literal_loop_rate()
    return {"value": pairs / secs, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "%d x 10 cm-1 windows of cfg2 (%.3g pairs, %.1f s) with the oracle's numpy slice-add restatement of "
                      "Isotope.createCrossSection; the reference's literal per-element Python loop runs at %.3g pairs/s "
                      "on the same core" % (k, pairs, secs, lit)}


def reference_arm(args, out):
    """--impl reference: the reference's CPU algorithm (oracle port; the reference itself is Python that cannot
    travel to the GPU box) on all host cores; each step = one 10 cm-1 cfg2 window per core."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        def step(s):
            jobs = [(1000.0 + 10.0 * ((s * cores + c) % 180), 10.0, 1000 + s * cores + c) for c in range(cores)]
            t0 = time.perf_counter()
            res = pool.map(_oracle_window, jobs)
            return sum(r[0] for r in res), time.perf_counter() - t0
        for s in range(args.warmup):
            step(s)
        pairs, secs = 0, 0.0
        for s in range(args.steps):
            p, t = step(args.warmup + s)
            pairs += p
            secs += t
    value = pairs / secs
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "impl": "reference",
        "config": {"workload": WORKLOAD, "sample": "each step: one 10 cm-1 window of the cell per host core"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "oracle numpy slice-add restatement of pyradClasses.py:361-400 (bitwise-equivalent "
                                   "order, ~15x faster than the reference's literal loop), %d processes, %d steps x %d "
                                   "windows of 10 cm-1" % (cores, args.steps, cores)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=out, flush=True)
    return 0


# ---------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N > 1: how the finished spectra are all-gathered -- 'peer' = stores into every rank's buffer "
                         "over NVLink from inside the compute kernel (default), 'nccl' = a separate NCCL all-gather")
    ap.add_argument("--no-atmosphere", action="store_true", help="skip the secondary 100-layer atmosphere object")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-farfield", action="store_true", help="skip the secondary far-field (PRB_K2_FARFIELD) measurements")
    ap.add_argument("--atm-layers", type=int, default=100)
    ap.add_argument("--atm-lines", type=int, default=5_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the transmittance and radiance spectra of the last timed step (the radiance above 0 cm-1, "
                         "where Planck's law is 0/0) as DIR/<name>.npy (float32; a fixed seeded sample of positions when "
                         "they exceed 64 MB), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm keeps no outputs (it measures a rate on sample windows)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    out = claim_stdout()
    if args.impl == "reference":
        return reference_arm(args, out)

    import torch
    import torch.distributed as dist
    from pyrad_b200 import distributed as pd
    from pyrad_b200 import engine as eng
    from pyrad_b200 import workloads

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with: python -m torch.distributed.run --nnodes=1 --nproc-per-node %d "
                             "--master-addr 127.0.0.1 --master-port P bench.py --gpus %d ..." % (args.gpus, args.gpus))
    numa = pin_rank_to_gpu_numa(local)              # before any pinned allocation (first touch decides the NUMA node)
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks, peaks_kind = load_peaks()

    # ------------------------------------------------------------------ workload (resident in HBM)
    w = workloads.cfg2_shard(rank, world)
    sp = w["species"]
    e = eng.Engine(local)
    # roofline denominators measured on THIS device, now (FFMA2 / FFMA instruction streams, float4 copy)
    measured = e.measure_peaks()
    e.upload_lines(w["lines"], n_groups=len(sp))
    e.set_grid(w["range_min"], w["res"], w["n_total"], w["i_begin"], w["i_end"])
    n_chunk = e.n_chunk
    T, P = w["T"], w["P"]
    win = eng.window_len(w["cutoff"], w["res"])
    molmass = [s.molmass for s in sp]
    q296 = [s.q296 for s in sp]
    qt = [[s.q(T) for s in sp]]
    conc = [w["conc"]]

    ext = torch.cuda.ExternalStream(e.stream)
    torch.cuda.set_stream(ext)                      # torch work (L2 flush, NCCL sync, events) follows the engine stream
    flush_buf = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")   # 512 MiB > 126 MB L2
    hold = {"gather": None}

    use_peer = world > 1 and args.gather == "peer"
    if use_peer:
        pd.connect_peers(e, rank, world, n_chunk, dist)

    # the step's C-ABI call with its (constant) arguments marshalled once: ~75 us of numpy / ctypes conversions per call
    # otherwise sit between the step's first event and its first kernel whenever the host is slower than the L2 flush
    step_call = e.atmosphere_call([w["depth_cm"]], [T], [P], conc, molmass, qt, q296, [win], w["t_surface"], w["range_max"])

    def step_device():
        """K1 -> K2 (layer physics fused into its epilogue) on resident inputs, and the all-gather of the finished
        radiance + transmittance spectra: peer stores from inside K2 + one flag barrier, or a separate NCCL call."""
        step_call()
        if world > 1 and not use_peer:
            rad_ptr, tr_ptr = e.atmosphere_result_dev()
            if hold["gather"] is None:
                hold["gather"] = [torch.empty(world * n_chunk, dtype=torch.float32, device="cuda") for _ in range(2)]
            dist.all_gather_into_tensor(hold["gather"][0], pd.device_tensor(rad_ptr, n_chunk))
            dist.all_gather_into_tensor(hold["gather"][1], pd.device_tensor(tr_ptr, n_chunk))

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # pair count of one step on this rank (exact, int64, computed by the library from the device's own indices)
    e.layer_prepass(T, P, conc[0], molmass, qt[0], q296, win)
    pairs_rank = e.pair_count()
    pairs_all = pairs_rank
    if world > 1:
        t = torch.tensor([pairs_rank], dtype=torch.int64, device="cuda")
        dist.all_reduce(t)
        pairs_all = int(t.item())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                 # sampled from warm-up through the timed region to the K2-only loop
    for _ in range(args.warmup):
        flush_buf.zero_()
        step_device()
    sync_all()
    # ---- timed region: K steps, CUDA events on the launching stream around every step, L2 flushed between steps
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sync_all()
    wall0 = time.perf_counter()
    for a, b in evs:
        flush_buf.zero_()
        a.record(ext)
        step_device()
        b.record(ext)
    sync_all()
    wall = time.perf_counter() - wall0
    if args.dump_outputs:
        outputs = step_outputs(e, n_chunk, world, dist, w["range_min"])   # before anything overwrites the result buffers
        if rank == 0:
            dump_outputs(args.dump_outputs, outputs)
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    launches_per_step = e.atmosphere_launches()
    headline_parity = None
    if use_peer:
        chunks = [(r * n_chunk, (r + 1) * n_chunk) for r in range(world)]
        headline_parity = gather_parity(e, chunks, n_chunk, rank, world, dist)
    tm = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    dev_ms = float(tm.item())
    ms_per_step = dev_ms / args.steps
    value = pairs_all / (ms_per_step * 1e-3)

    # ---- dominant kernel alone (K2) for the roofline: events around prb_line_sum_dev only, L2 flushed
    kbuf = torch.empty(n_chunk, dtype=torch.float32, device="cuda")
    wts = [eng.number_density_weight(c, P, T) for c in w["conc"]]
    e.layer_prepass(T, P, conc[0], molmass, qt[0], q296, win, wts)
    k2_ms = []
    for i in range(3 + 10):
        flush_buf.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(ext)
        e.line_sum_dev(kbuf.data_ptr(), eng.OUT_F32)
        b.record(ext)
        torch.cuda.synchronize()
        if i >= 3:
            k2_ms.append(a.elapsed_time(b))
    k2_t = float(np.mean(k2_ms)) * 1e-3
    clocks = sampler.stop() if rank == 0 else None

    # ---- e2e: the same step through the C ABI with HOST buffers (pinned), copies inside the timed region
    host_lines = {}
    for kname, v in w["lines"].items():
        tns = torch.from_numpy(np.ascontiguousarray(v)).pin_memory()
        host_lines[kname] = tns.numpy()
        host_lines["_keep_" + kname] = tns
    h_rad = torch.empty(n_chunk, dtype=torch.float32).pin_memory()
    h_tr = torch.empty(n_chunk, dtype=torch.float32).pin_memory()
    lines_view = {k: v for k, v in host_lines.items() if not k.startswith("_keep_")}

    e.set_result_host(h_rad.numpy(), h_tr.numpy())     # zero-copy delivery: K2's epilogue stores into these pinned buffers

    e2e_call = e.gas_cell_host_call(lines_view, len(sp), w["range_min"], w["res"], w["n_total"], w["i_begin"], w["i_end"],
                                    w["depth_cm"], T, P, conc[0], molmass, qt[0], q296, win, w["t_surface"], w["range_max"])

    def step_e2e():
        # ONE call, host buffers in, host buffers out: the line columns cross PCIe in wavenumber pieces while the
        # earlier pieces' prepass and line sums already run (H2D), finished tiles land in h_rad / h_tr (D2H)
        e2e_call()
        if world > 1 and not use_peer:
            rad_ptr, tr_ptr = e.atmosphere_result_dev()
            dist.all_gather_into_tensor(hold["gather"][0], pd.device_tensor(rad_ptr, n_chunk))
            dist.all_gather_into_tensor(hold["gather"][1], pd.device_tensor(tr_ptr, n_chunk))

    for _ in range(2):
        step_e2e()
    sync_all()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    sync_all()
    e2e_s = time.perf_counter() - t0
    e.set_result_host()
    # the same call from ORDINARY (pageable) numpy arrays, results copied out into pageable float32 arrays: what a caller
    # gets who hands over whatever numpy gave them (the copies then go through the driver's staging buffer)
    pageable_ms = None
    if world == 1:
        plain_lines = {k: np.array(v) for k, v in w["lines"].items()}
        p_rad, p_tr = np.empty(n_chunk, dtype=np.float32), np.empty(n_chunk, dtype=np.float32)
        plain_call = e.gas_cell_host_call(plain_lines, len(sp), w["range_min"], w["res"], w["n_total"], w["i_begin"], w["i_end"],
                                          w["depth_cm"], T, P, conc[0], molmass, qt[0], q296, win, w["t_surface"], w["range_max"])

        def step_plain():
            plain_call()
            e.atmosphere_read_f32(p_rad, p_tr)
        for _ in range(2):
            step_plain()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            step_plain()
        pageable_ms = (time.perf_counter() - t0) / e2e_steps * 1e3
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    n_l = e.n_lines
    h2d = n_l * (7 * 8 + 4) + 4 * 32 * len(sp)
    d2h = 4 * (n_l + 20) + 2 * 4 * n_chunk + 16 * 8
    e2e = {"value": pairs_all / (e2e_s / e2e_steps), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_s / e2e_steps * 1e3, "pageable_ms_per_step": pageable_ms,
           "api": "prb_gas_cell_host with prb_set_result_host: pinned host buffers in and out, line columns uploaded in wavenumber pieces under the compute, results stored into host memory tile by tile from inside K2"}

    # ---- secondary object: the same cell with the opt-in far-field variant of K2 (Lorentz wings of far lines summed at
    # 8 Chebyshev nodes per warp span and interpolated; DESIGN.md).  The headline above is the exact per-point kernel.
    far = None
    if not args.no_farfield:
        k_exact = torch.empty(n_chunk, dtype=torch.float64, device="cuda")
        k_far = torch.empty(n_chunk, dtype=torch.float64, device="cuda")
        e.layer_prepass(T, P, conc[0], molmass, qt[0], q296, win, wts)
        e.line_sum_dev(k_exact.data_ptr(), eng.OUT_F64)
        e.set_k2_variant(eng.K2_FARFIELD, 0)
        try:
            e.layer_prepass(T, P, conc[0], molmass, qt[0], q296, win, wts)
            e.line_sum_dev(k_far.data_ptr(), eng.OUT_F64)
            torch.cuda.synchronize()
            floor = 1e-40 * float(k_exact.abs().max().item())
            rel = float(((k_far - k_exact).abs() / torch.clamp(k_exact.abs(), min=floor)).max().item())
            fk2 = []
            for i in range(3 + 10):
                flush_buf.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(ext)
                e.line_sum_dev(kbuf.data_ptr(), eng.OUT_F32)
                b.record(ext)
                torch.cuda.synchronize()
                if i >= 3:
                    fk2.append(a.elapsed_time(b))
            fsteps = max(3, min(args.steps, 50))
            for _ in range(3):
                flush_buf.zero_()
                step_device()
            sync_all()
            fev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(fsteps)]
            for a, b in fev:
                flush_buf.zero_()
                a.record(ext)
                step_device()
                b.record(ext)
            sync_all()
            tf = torch.tensor([sum(a.elapsed_time(b) for a, b in fev) / fsteps], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tf, op=dist.ReduceOp.MAX)
            far_ms = float(tf.item())
            e.set_result_host(h_rad.numpy(), h_tr.numpy())
            for _ in range(2):
                step_e2e()
            sync_all()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                step_e2e()
            sync_all()
            te = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device="cuda")
            e.set_result_host()
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            far = {"variant": FARFIELD_NOTE + " -- NOT the headline: value / e2e / roofline are the exact per-point kernel",
                   "k2_ms": float(np.mean(fk2)), "k2_equivalent_pairs_per_s": pairs_rank / (float(np.mean(fk2)) * 1e-3),
                   "ms_per_step": far_ms, "equivalent_pairs_per_s": pairs_all / (far_ms * 1e-3),
                   "e2e_ms_per_step": float(te.item()) * 1e3, "e2e_equivalent_pairs_per_s": pairs_all / float(te.item()),
                   "max_rel_diff_of_k_vs_exact_kernel": rel, "steps": fsteps}
            try:
                # what the far-field kernel really evaluates on this rank's chunk (host-side restatement of its integer
                # class tests, tests/test_partition.py): pairs evaluated point by point + node evaluations, and the
                # FP32 lane-slots they cost (13 packed instructions per 6 pairs, 19 per 12 node evaluations), against the
                # measured FFMA2 rate
                from pyrad_b200 import partition as pt
                ex_pairs, node_evals = pt.farfield_work(pt.line_index(w["lines"]["nu"], w["range_min"], w["res"]),
                                                        w["i_begin"], w["i_end"], win, 256)
                slots = ex_pairs * 13.0 / 3.0 + node_evals * 19.0 / 6.0
                peak_slots = measured["ffma2_lane_fma_per_s"]
                far["evaluated_pairs_this_rank"] = int(ex_pairs)
                far["node_evaluations_this_rank"] = int(node_evals)
                far["k2_fp32_lane_slot_frac"] = slots / (far["k2_ms"] * 1e-3) / peak_slots
            except Exception as exc:                      # accounting only: never let it cost the bench line
                far["work_accounting_error"] = repr(exc)
        finally:
            e.set_k2_variant(eng.K2_CLASSED, 0)

    # ---- secondary object: the 100-layer atmosphere (cfg4), strong-sharded by wavenumber chunk
    atm = None
    if not args.no_atmosphere:
        atm = run_atmosphere(e, args, rank, world, ext, peaks, use_peer)

    # ---- secondary object: the cfg5 stress sweep (5M lines, 5M points, 25 cm-1 cutoff), strong-sharded like the atmosphere
    stress = None
    if not args.no_atmosphere:
        stress = run_stress(e, rank, world, ext, use_peer, not args.no_farfield)

    # ---- secondary objects at N = 1: the other BASELINE gas cells (cfg1, cfg3) through the one-call path, the host
    # mirror on cfg2, line-list ingestion (section 8(f) row 1)
    ingest = small = mirror = None
    if rank == 0 and world == 1:
        from pyrad_b200 import workloads as wl
        small = {"cfg1": run_small_cell(e, ext, wl.cfg1(), "cfg1: CO2 cell 500-800 cm-1 @ 0.01 cm-1 (30 000 points, 50k lines, W = 500)", flush_buf),
                 "cfg3": run_small_cell(e, ext, wl.cfg3(), "cfg3: CO2 + H2O line by line + CFC-11 / HCFC-22 xsc tables, 500-800 cm-1 @ 0.01 cm-1", flush_buf)}
        try:
            # the REAL reference on this very workload, timed in the build container where its sources are mounted
            # (scripts/time_reference_cfg1.py; committed next to the goldens): same inputs, same pair count
            real = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_cfg1_timing.json")))
            if real["pairs"] == small["cfg1"]["pairs"]:
                small["cfg1"]["reference_real"] = {
                    "get_transmittance_s": real["get_transmittance_s"], "pairs_per_s": real["pairs_per_s"], "cores": 1,
                    "machine": real["machine"], "what": real["what"],
                    "e2e_speedup_vs_real_reference": real["get_transmittance_s"] * 1e3 / small["cfg1"]["e2e"]["ms_per_step"]}
        except Exception:
            pass
        mirror = run_mirror(e, w, e2e["ms_per_step"])
    if rank == 0 and world == 1 and not args.no_cpu:
        ingest = run_ingest(e, w)

    # ---- CPU baseline (rank 0, N = 1 only): oracle port on a bounded sample of the same workload
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline_sample()

    if rank == 0:
        sm_max = float(peaks.get("sm_max_mhz", SM_MAX_MHZ_DEFAULT))
        f_hz = sm_max * 1e6
        # FP32-pipe roofline of K2, the pipe that binds the triple-reciprocal formulation (ncu: math_pipe_throttle is
        # the top stall, pipe_fma_cycles_active ~70 %).  Denominator: the FFMA2 lane-FMA rate MEASURED on this device a
        # minute ago (prb_measure_peaks; the nominal 148 SM x 128 lanes x f_max is printed beside it).  Numerator, two
        # ways: what this kernel executes -- 13 packed FP32x2 instructions per six (line, point) pairs = 4.33 lane-slots
        # per pair -- and the leanest formulation measured (A-normalised triple, 11 packed = 3.67; scripts/ubench/triple.cu).
        fp32_nominal = SM_COUNT * 128 * 2 * f_hz / 1e12
        fp32_peak = measured["ffma2_lane_fma_per_s"] * 2 / 1e12
        k2_pairs_s = pairs_rank / k2_t
        slots_per_pair, slots_min = 13.0 / 3.0, 11.0 / 3.0
        fp32_ach = k2_pairs_s * slots_per_pair * 2 / 1e12
        mufu_naive_peak = SM_COUNT * 16 * f_hz / 2.0          # SURVEY 8(d): 2 MUFU per Voigt pair
        hbm_measured = measured["copy_bytes_per_s"] / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "parallelism": "wavenumber chunks x%d, %s" % (
                           world, "no collective" if world == 1 else
                           ("all-gather fused into K2 (NVLink peer stores + flag barrier)" if use_peer else "NCCL all-gather")),
                       "pairs_per_step": pairs_all, "lines_per_gpu": n_l, "points_per_gpu": n_chunk,
                       "l2": "flushed between timed steps (512 MiB write)",
                       "numerics": "FP64 prepass, FP32 lineshape evaluation, FP64 accumulation; k stored FP32",
                       "host_affinity": numa},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * args.steps,
            "gather_parity": headline_parity,
            "roofline": {"bound": "fp32", "achieved": fp32_ach, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": fp32_ach / fp32_peak, "frac_minimum_formulation": k2_pairs_s * slots_min * 2 / 1e12 / fp32_peak,
                         "traffic": load_traffic("k2_line_sum<8>@cfg2"),
                         "traffic_unit": "DRAM bytes per launch (ncu --set full, profiles/traffic.json); the kernel is FP32-pipe "
                                         "bound, its algorithmic DRAM traffic is the 18 MB of line records",
                         "kernel": "k2_line_sum<8>",
                         "k2_ms": k2_t * 1e3, "k2_pairs_per_s": k2_pairs_s,
                         "peak_source": "measured",
                         "peak_how": "prb_measure_peaks in this run: packed FFMA2 stream %.2f TFLOP/s (scalar FFMA stream %.2f; nominal "
                                     "148 SM x 128 lanes x 2 x %.0f MHz = %.2f); float4 copy %.0f GB/s (MEASURED_PEAKS.json %s: %.0f)" % (
                                         fp32_peak, measured["ffma_lane_fma_per_s"] * 2 / 1e12, sm_max, fp32_nominal, hbm_measured,
                                         peaks_kind, float(peaks.get("hbm_gbs", 0.0))),
                         "algorithmic": "frac: 4.33 FP32 lane-slots (x2 flop) per (line, gridpoint) pair = what k2_line_sum executes "
                                        "(13 packed FP32x2 instr per 6 pairs, DESIGN.md section 4); frac_minimum_formulation: 3.67 "
                                        "(11 packed, the leanest variant measured); real flops are 6.33 per pair"},
            "roofline_sfu": {"bound": "sfu", "achieved": k2_pairs_s / 1e9, "peak": mufu_naive_peak / 1e9, "unit": "Gpair/s",
                             "frac": k2_pairs_s / mufu_naive_peak,
                             "note": "SURVEY 8(d) naive bound (2 MUFU per Voigt pair, 16 MUFU/clk/SM); the kernel issues "
                                     "1/3 MUFU per Lorentz pair (triple reciprocal), hence > 1"},
            "measured_peaks": measured,
            "wall_s_timed_region": wall,
        }
        # the 1 -> 8 curves of the strong-scaled objects, readable without walking the nested objects
        if atm:
            line["atmosphere_ms"] = atm["ms_per_spectrum"]
            line["atmosphere_exact_ms"] = atm["exact_kernel"]["ms_per_spectrum"]
            line["atmosphere_spectra_per_s"] = atm["spectra_per_s"]
        if stress:
            line["stress_ms"] = stress["ms"]
            line["stress_exact_ms"] = stress["exact_kernel"]["ms"]
        if small:
            line["cfg1"] = small["cfg1"]
            line["cfg3"] = small["cfg3"]
        if mirror:
            line["mirror"] = mirror
        if far:
            line["farfield"] = far
        if atm:
            line["atmosphere"] = atm
        if stress:
            line["stress_sweep"] = stress
        if ingest:
            line["ingest"] = ingest
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), file=out, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_small_cell(e, ext, w, name, flush_buf, steps=50):
    """A BASELINE gas-cell configuration that is not the bench workload (cfg1: the reference's own CPU-runnable case;
    cfg3: line-by-line + xsc tables) through the same ONE-call path: device-timed steps on resident inputs, and the e2e
    call from pinned host buffers to pinned host buffers (for cfg3 the xsc tables are re-registered inside every e2e
    step: they are inputs too)."""
    import torch
    from pyrad_b200 import classes as C
    from pyrad_b200 import engine as eng
    sp = w["species"]
    n = eng.grid_len(w["range_min"], w["range_max"], w["res"])
    win = eng.window_len(w["cutoff"], w["res"])
    T, P = w["T"], w["P"]
    molmass, q296, qt = [s.molmass for s in sp], [s.q296 for s in sp], [s.q(T) for s in sp]
    xa = np.linspace(w["range_min"], w["range_max"], n, endpoint=True)
    plans = []
    for x in w.get("xsc", []):
        grid01 = np.arange(x["range_min"], x["range_max"], .01)
        dst0, src0, count, _ = C._merge_plan(xa, grid01)
        coarse = x["res"] > .01
        plans.append(dict(n_out=n, dst0=dst0, src0=src0, count=count, file_x=x["wavenumber"] if coarse else None,
                          file_y=x["intensity"], interp=coarse, ax0=float(grid01[0]), adelta=float(grid01[1] - grid01[0])))

    def register_tables():
        e.xsc_clear()
        for slot, pl in enumerate(plans):
            e.xsc_resident(slot, **pl)
        if plans:
            e.set_xsc_conc([[x["conc"] for x in w["xsc"]]])

    e.upload_lines(w["lines"], n_groups=len(sp))
    e.set_grid(w["range_min"], w["res"], n)
    register_tables()
    try:
        e.layer_prepass(T, P, w["conc"], molmass, qt, q296, win)
        pairs = e.pair_count()
        call = e.atmosphere_call([w["depth_cm"]], [T], [P], [w["conc"]], molmass, [qt], q296, [win], 288.0, w["range_max"])
        for _ in range(3):
            call()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        torch.cuda.synchronize()
        for a, b in evs:
            flush_buf.zero_()
            a.record(ext)
            call()
            b.record(ext)
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in evs) / steps
        launches = e.atmosphere_launches()
        host = {}
        keep = []
        for kname, v in w["lines"].items():
            tns = torch.from_numpy(np.ascontiguousarray(v)).pin_memory()
            keep.append(tns)
            host[kname] = tns.numpy()
        h_rad = torch.empty(n, dtype=torch.float32).pin_memory()
        h_tr = torch.empty(n, dtype=torch.float32).pin_memory()
        e.set_result_host(h_rad.numpy(), h_tr.numpy())
        cell = e.gas_cell_host_call(host, len(sp), w["range_min"], w["res"], n, 0, n, w["depth_cm"], T, P, w["conc"], molmass,
                                    qt, q296, win, 288.0, w["range_max"])

        def e2e_step():
            if plans:
                register_tables()
            cell()
        for _ in range(2):
            e2e_step()
        e.synchronize()
        reps = 10
        t0 = time.perf_counter()
        for _ in range(reps):
            e2e_step()
        e.synchronize()
        e2e_ms = (time.perf_counter() - t0) / reps * 1e3
        e.set_result_host()
        n_l = len(w["lines"]["nu"])
        xsc_bytes = sum(8 * len(x["intensity"]) * (2 if x["res"] > .01 else 1) for x in w.get("xsc", []))
        return {"workload": name, "pairs": pairs, "points": n, "lines": n_l, "xsc_tables": len(plans),
                "ms_per_step": ms, "pairs_per_s": pairs / (ms * 1e-3), "launches_per_step": launches,
                "e2e": {"ms_per_step": e2e_ms, "value": pairs / (e2e_ms * 1e-3), "unit": UNIT,
                        "h2d_bytes_per_step": int(n_l * (7 * 8 + 4) + xsc_bytes), "d2h_bytes_per_step": int(2 * 4 * n),
                        "api": "prb_gas_cell_host (+ prb_xsc_resident per table) with prb_set_result_host, pinned buffers"},
                "mean_transmittance": float(np.nanmean(h_tr.numpy()))}
    finally:
        e.xsc_clear()


def run_mirror(e, w, e2e_ms):
    """The reference-facing object model itself (pyrad_b200/classes.py: Layer > Molecule > Isotope) on cfg2 with ordinary
    PAGEABLE numpy line arrays attached to the isotopologues: getTransmittance(layer) from a cold layer (cross sections
    reset before every call), i.e. grouped upload + grid index + prepass + one line-sum launch with a row per isotopologue
    + k -> T on the device + the FP64 transmittance back to the host.  Also: the per-isotopologue rows ("layer and
    components" plots, pyradClasses.py:566-576) and how long building the objects takes."""
    import shutil
    import tempfile
    from pyrad_b200 import classes as C
    root = tempfile.mkdtemp(prefix="prb_mirror_")
    old = (C.DATA_ROOT, C.BASE_RESOLUTION, C.Layer.hasAtmosphere, C._ENGINE)
    try:
        for s in w["species"]:                                   # the two small per-isotopologue files the constructors read
            d = os.path.join(root, "data", str(s.global_iso))
            os.makedirs(d)
            with open(os.path.join(d, "params.pyr"), "w") as f:
                f.write("# params\n%d,%s,%d,1,0.99,%r,1,%r\n" % (s.global_iso, s.name, s.mol_id, float(s.q296), float(s.molmass)))
        C.set_engine(e)
        C.DATA_ROOT, C.BASE_RESOLUTION, C.Layer.hasAtmosphere = root, w["res"], False
        t0 = time.perf_counter()
        layer = C.Layer(w["depth_cm"], w["T"], w["P"], w["range_min"], w["range_max"], dynamicResolution=False)
        for g, (s, c) in enumerate(zip(w["species"], w["conc"])):
            m = C.Molecule(s.name, layer, concentration=c)
            layer.append(m)
            m[0].setLines({k: np.array(v) for k, v in w["per_group_lines"][g].items()}, {int(w["T"]): s.q(w["T"])})
        build_ms = (time.perf_counter() - t0) * 1e3
        n_lines = sum(len(m[0]) for m in layer)

        def cold_transmittance():
            C.resetCrossSection(layer)
            C._RESIDENT_KEY = None
            return C.getTransmittance(layer)
        # the first calls also page-lock the result arrays the mirror's pool then reuses (engine.ResultPool: ~15 ms per
        # 24 MB block, once per result size); the figure quoted is the steady state of a session that recomputes a layer
        t0 = time.perf_counter()
        tr = cold_transmittance()
        first_ms = (time.perf_counter() - t0) * 1e3
        for _ in range(2):
            tr = cold_transmittance()
        reps = 5
        t0 = time.perf_counter()
        for _ in range(reps):
            tr = cold_transmittance()
        cold_ms = (time.perf_counter() - t0) / reps * 1e3
        t0 = time.perf_counter()
        rows = [C.getCrossSection(m[0]) for m in layer]          # the rows are still on the device: one D2H for all four
        comp_ms = (time.perf_counter() - t0) * 1e3
        # where the cold call's time goes: the same engine calls, one by one (host wall clock, synchronised)
        isos = [m[0] for m in layer]
        stage = {}

        def lap(name, fn):
            e.synchronize()
            t = time.perf_counter()
            out = fn()
            e.synchronize()
            stage[name] = (time.perf_counter() - t) * 1e3
            return out
        n_pts = len(tr)
        win = eng_window = None
        from pyrad_b200 import engine as eng
        win = eng.window_len(layer.distanceFromCenter, layer.resolution)
        lap("upload_line_groups_ms", lambda: e.upload_line_groups([iso._cols for iso in isos]))
        lap("set_grid_ms", lambda: e.set_grid(layer.rangeMin, layer.resolution, n_pts))
        lap("layer_prepass_ms", lambda: e.layer_prepass(layer.T, layer.P, [iso.molecule.concentration for iso in isos],
                                                        [iso.molmass for iso in isos], [iso.q[layer.T] for iso in isos],
                                                        [iso.q296 for iso in isos], win))
        lap("line_sum_groups_ms", lambda: e.line_sum_groups(to_host=False))
        wts = [eng.number_density_weight(iso.molecule.concentration, layer.P, layer.T) for iso in isos]
        lap("layer_spectra_resident_ms", lambda: e.layer_spectra_resident(wts, layer.depth, layer.T, layer.rangeMax,
                                                                          want=("transmittance",)))
        C._RESIDENT_KEY = None
        return {"workload": "cfg2 through pyrad_b200.classes (Layer > Molecule > Isotope), pageable numpy line arrays, float64 results",
                "lines": n_lines, "points": len(tr), "build_objects_ms": build_ms,
                "get_transmittance_cold_ms": cold_ms, "first_call_ms": first_ms, "vs_c_abi_e2e": cold_ms / e2e_ms if e2e_ms else None,
                "per_isotopologue_rows_ms": comp_ms, "rows": len(rows), "cold_call_stages": stage,
                "bytes": {"h2d": int(n_lines * 7 * 8), "d2h_transmittance": int(8 * len(tr)), "d2h_rows": int(8 * len(tr) * len(rows))},
                "mean_transmittance": float(np.nanmean(tr)),
                "api": "classes.getTransmittance(layer): prb_upload_line_groups + prb_set_grid + prb_layer_prepass + "
                       "prb_line_sum_groups + prb_layer_spectra_resident"}
    finally:
        C.DATA_ROOT, C.BASE_RESOLUTION, C.Layer.hasAtmosphere = old[0], old[1], old[2]
        C.set_engine(old[3])
        shutil.rmtree(root, ignore_errors=True)


def run_ingest(e, w):
    """HITRAN-online CSV text of the cfg2 line list -> device SoA (K5 parser) versus the reference's reader
    (oracle restatement of readHitranOnlineFile) on a bounded sample of the same rows."""
    from oracle import physics as ph
    ln = w["lines"]
    n = len(ln["nu"])
    cols = [ln[k] for k in ("nu", "sw", "gamma_air", "gamma_self", "elower", "n_air", "delta_air")]
    t0 = time.perf_counter()
    rows = ["2,1,%r,%r,1.0,%r,%r,%r,%r,%r" % (float(a), float(b), float(el), float(ga), float(gs), float(d), float(na))
            for a, b, ga, gs, el, na, d in zip(*cols)]
    text = ("\n".join(rows) + "\n").encode()
    fmt_s = time.perf_counter() - t0
    lo, hi = -1.0, 1e9
    e.ingest_csv(text, lo, hi)                       # warm-up (allocations)
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        kept = e.ingest_csv(text, lo, hi)
    dev_s = (time.perf_counter() - t0) / reps
    sample = rows[: min(n, 60000)]
    t0 = time.perf_counter()
    ref = ph.read_hitran_online_rows(sample, lo, hi)
    cpu_s = time.perf_counter() - t0
    got = e.download_lines()
    ok = bool(np.array_equal(got["nu"][: len(ref["nu"])], ref["nu"]) and np.array_equal(got["sw"][: len(ref["sw"])], ref["sw"]))
    return {"workload": "cfg2 line list as HITRAN-online CSV text (%d rows, %.1f MB)" % (n, len(text) / 1e6),
            "lines_per_s": kept / dev_s, "ms": dev_s * 1e3, "text_gb_per_s": len(text) / dev_s / 1e9,
            "api": "prb_ingest_hitran_csv (pageable host text in, device SoA out; H2D copy inside the timed region)",
            "cpu_reference_lines_per_s": len(sample) / cpu_s, "cpu_sample_rows": len(sample), "bit_exact_vs_cpu": ok,
            "host_text_formatting_s": fmt_s}


def run_sharded_column(e, w, windows, column_args, rank, world, ext, use_peer, variant, reps, want_timing=False):
    """One spectrum of a column workload strong-sharded over the ranks by wavenumber chunk, with K2 variant `variant`:
    plan on the variant's own cost model, place, one warm-up run, ONE feedback step of the cuts from the per-rank device
    times (N > 1), then `reps` timed runs (CUDA events on the engine stream, barrier + synchronise around each, max over
    ranks of the median).  Returns the measurements, and -- N > 1 with the peer gather -- the bitwise comparison of the
    gather buffer with a separate NCCL all-gather."""
    import torch
    import torch.distributed as dist
    from pyrad_b200 import distributed as pd
    from pyrad_b200 import engine as eng

    sp = w["species"]
    n_total = eng.grid_len(w["range_min"], w["range_max"], w["res"])
    far = variant == eng.K2_FARFIELD
    state = {}

    def place(p):
        """(Re)load this rank's share of plan p: its lines, its chunk, its slot of the peer gather buffers."""
        e.upload_lines(p.subset(w["lines"]), n_groups=len(sp))
        e.set_grid(w["range_min"], w["res"], n_total, p.i_begin, p.i_end)
        if use_peer:
            e.peer_disconnect()
            pd.connect_peers(e, rank, world, p.max_chunk, dist)
        state["plan"], state["nc"] = p, p.i_end - p.i_begin

    def run():
        p, nc = state["plan"], state["nc"]
        e.atmosphere(*column_args)
        if world > 1 and not use_peer:
            rad_p, tr_p = e.atmosphere_result_dev()
            pd.all_gather_spectra(pd.device_tensor(rad_p, nc), p, dist)
            pd.all_gather_spectra(pd.device_tensor(tr_p, nc), p, dist)

    e.set_k2_variant(variant, 0)
    e.set_timing(True)
    # strong scaling over small chunks: short K2 launches hand every tile out as line-range parts (no idle last wave)
    e.set_option(eng.OPT_SPLIT_TILES, 1 if world > 1 else 0)
    try:
        place(pd.ShardPlan(w["lines"]["nu"], w["range_min"], w["res"], n_total, windows, rank, world, farfield=far))
        for _ in range(2 if world > 1 else 1):          # (the first run allocates; the feedback step reads a warm one)
            run()
            torch.cuda.synchronize()
        rebalanced = False
        if world > 1:
            def slowest_rank_ms():
                t = e.atmosphere_timing()
                mine = torch.tensor([t["k1_ms"] + t["k2_ms"] + t["k3_ms"]], dtype=torch.float64, device="cuda")
                allt = torch.empty(world, dtype=torch.float64, device="cuda")
                dist.all_gather_into_tensor(allt, mine)
                return [float(x) for x in allt.tolist()]
            before = slowest_rank_ms()
            plan1 = state["plan"]
            plan2 = plan1.rebalanced(before)
            if plan2 is not plan1:
                place(plan2)
                for _ in range(2):
                    run()
                    torch.cuda.synchronize()
                after = slowest_rank_ms()
                # the feedback step is linear in the chunk's cost; a launch of a few waves is a step function of its tile
                # count, so the moved cuts are kept only if the slowest rank really got faster
                if max(after) < max(before):
                    rebalanced = True
                else:
                    place(plan1)
                    run()
                    torch.cuda.synchronize()
            dist.barrier()
        times = timed_runs(ext, run, reps, world, dist)
        tim = e.atmosphere_timing()
        ms, k1, k2, k3 = max_over_ranks([float(np.median(times)), tim["k1_ms"], tim["k2_ms"], tim["k3_ms"]], world, dist)
        parity = gather_parity(e, state["plan"].chunks, state["nc"], rank, world, dist) if (world > 1 and use_peer) else None
        return {"ms": ms, "ms_runs_this_rank": [float(t) for t in times], "rank0_stage_ms": tim,
                "max_rank_stage_ms": {"k1_ms": k1, "k2_ms": k2, "k3_ms": k3}, "launches": e.atmosphere_launches(),
                "chunk_points_rank0": state["nc"], "rebalanced": rebalanced, "gather_parity": parity,
                "split_tiles": world > 1}
    finally:
        e.set_timing(False)
        e.set_option(eng.OPT_SPLIT_TILES, 0)
        e.set_k2_variant(eng.K2_CLASSED, 0)


FARFIELD_NOTE = ("K2 variant PRB_K2_FARFIELD: Lorentz wings of lines farther than one span length from a warp's 128/256-point "
                 "span (and covering it fully) are summed at 16 Chebyshev nodes of the span and interpolated once per tile "
                 "-- for windows of four tile lengths and more, lines far from the whole 2048-point tile once per tile; "
                 "interpolation error <= 2e-8 of k (FP64 model, tests/test_farfield_model.py); every pair's contribution is "
                 "in the result, far pairs are not evaluated one by one")


def run_stress(e, rank, world, ext, use_peer, farfield=True):
    """cfg5: one gas cell, 5M synthetic lines, 0-5000 cm-1 @ 0.001 cm-1, fixed 25 cm-1 cutoff (W = 25 000, ~2.5e11
    accumulations), split over the N ranks by wavenumber chunk; the finished spectra gathered as in the headline.
    The object's default is the far-field variant of K2 (spectra/s is not a pair count); the exact per-point kernel --
    the one the line-gridpoint headline is measured on -- is timed beside it."""
    from pyrad_b200 import engine as eng
    from pyrad_b200 import partition as pt
    from pyrad_b200 import workloads

    w = workloads.cfg5()
    sp = w["species"]
    n_total = eng.grid_len(w["range_min"], w["range_max"], w["res"])
    win = eng.window_len(w["cutoff"], w["res"])
    T, P = w["T"], w["P"]
    args_ = ([w["depth_cm"]], [T], [P], [w["conc"]], [s.molmass for s in sp], [[s.q(T) for s in sp]], [s.q296 for s in sp],
             [win], 288.0, w["range_max"])
    exact = run_sharded_column(e, w, [win], args_, rank, world, ext, use_peer, eng.K2_CLASSED, 3)
    far = run_sharded_column(e, w, [win], args_, rank, world, ext, use_peer, eng.K2_FARFIELD, 3) if farfield else None
    idx = np.trunc((w["lines"]["nu"] - w["range_min"]) / w["res"]).astype(np.int64)
    pairs = float(pt.block_pair_cost(idx, n_total, [win]).sum())
    out = {"workload": "cfg5: 5M synthetic lines, 0-5000 cm-1 @ 0.001 cm-1 (%d points), fixed 25 cm-1 cutoff (W = %d)" % (n_total, win),
           "pairs": pairs, "scaling": "strong", "n_gpus": world,
           "exact_kernel": {"ms": exact["ms"], "pairs_per_s": pairs / (exact["ms"] * 1e-3),
                            "ms_runs_this_rank": exact["ms_runs_this_rank"], "gather_parity": exact["gather_parity"]}}
    head = far or exact
    out.update({"ms": head["ms"], "spectra_per_s": 1e3 / head["ms"], "ms_runs_this_rank": head["ms_runs_this_rank"],
                "equivalent_pairs_per_s": pairs / (head["ms"] * 1e-3), "gather_parity": head["gather_parity"],
                "k2_variant": FARFIELD_NOTE if far else "PRB_K2_CLASSED (exact per-point kernel)"})
    return out


def run_atmosphere(e, args, rank, world, ext, peaks, use_peer):
    """100-layer standard atmosphere, 0-5000 cm-1 @ 0.001 cm-1, ~5M lines: K1+K2 per layer, one K3 fold, one
    all-gather.  Strong scaling: the N ranks split ONE spectrum by wavenumber chunks balanced on the kernel's cost model.
    Default variant of this object: far-field K2; the exact per-point kernel is timed beside it."""
    from pyrad_b200 import engine as eng
    from pyrad_b200 import partition as pt
    from pyrad_b200 import workloads

    w = workloads.atmosphere(n_layers=args.atm_layers, n_lines=args.atm_lines)
    sp = w["species"]
    n_total = eng.grid_len(w["range_min"], w["range_max"], w["res"])
    win = [eng.window_len(c, w["res"]) for c in w["cutoff"]]
    qt = np.array([[s.q(T) for s in sp] for T in w["T"]])
    col = (w["depth_cm"], w["T"], w["P"], w["conc"], [s.molmass for s in sp], qt, [s.q296 for s in sp], win,
           w["t_surface"], w["range_max"])
    exact = run_sharded_column(e, w, win, col, rank, world, ext, use_peer, eng.K2_CLASSED, 5)
    far = run_sharded_column(e, w, win, col, rank, world, ext, use_peer, eng.K2_FARFIELD, 5) if not args.no_farfield else None
    idx = np.trunc((w["lines"]["nu"] - w["range_min"]) / w["res"]).astype(np.int64)
    pairs = float(pt.block_pair_cost(idx, n_total, win).sum())
    head = far or exact
    nc = head["chunk_points_rank0"]
    k3_bytes = len(win) * nc * 4 + nc * 8
    k1_bytes = len(w["lines"]["nu"]) / max(world, 1) * (56.0 + 36.0 * len(win))      # approx. per rank: columns once + records
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    k3_ms, k1_ms = head["rank0_stage_ms"]["k3_ms"], head["rank0_stage_ms"]["k1_ms"]
    out = {"workload": "cfg4: %d-layer US-std atmosphere 0-70 km, 0-5000 cm-1 @ 0.001 cm-1 (%d points, %d lines), "
                       "reference cutoff 5*P/p0 per layer" % (len(win), n_total, len(w["lines"]["nu"])),
           "k2_variant": FARFIELD_NOTE if far else "PRB_K2_CLASSED (exact per-point kernel)",
           "spectra_per_s": 1e3 / head["ms"], "ms_per_spectrum": head["ms"], "ms_runs_this_rank": head["ms_runs_this_rank"],
           "pairs": pairs, "equivalent_pairs_per_s": pairs / (head["ms"] * 1e-3),
           "scaling": "strong", "n_gpus": world, "chunk_points_rank0": nc, "launches": head["launches"],
           "partition": "measured-class-cost model of the variant" + (", one feedback step on the warm-up run's per-rank times" if head["rebalanced"] else ""),
           "gather": "none" if world == 1 else ("peer stores fused into K3" if use_peer else "nccl"),
           "gather_parity": head["gather_parity"],
           "rank0_stage_ms": head["rank0_stage_ms"], "max_rank_stage_ms": head["max_rank_stage_ms"],
           "exact_kernel": {"ms_per_spectrum": exact["ms"], "pairs_per_s": pairs / (exact["ms"] * 1e-3),
                            "ms_runs_this_rank": exact["ms_runs_this_rank"], "rank0_stage_ms": exact["rank0_stage_ms"],
                            "max_rank_stage_ms": exact["max_rank_stage_ms"], "gather_parity": exact["gather_parity"]},
           "roofline_k3": {"bound": "hbm", "achieved": k3_bytes / (k3_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                           "frac": k3_bytes / (k3_ms * 1e-3) / 1e9 / hbm,
                           "traffic": load_traffic("k3_fold_f32@cfg4") if world == 1 and len(win) == 100 else None,
                           "algorithmic_bytes": k3_bytes},
           "roofline_k1": {"bound": "hbm", "achieved": k1_bytes / (k1_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                           "frac": k1_bytes / (k1_ms * 1e-3) / 1e9 / hbm, "algorithmic_bytes": k1_bytes,
                           "note": "56 B of line columns once + 36 B of records per line-layer; the kernel is FP64-pipe / "
                                   "issue bound (DESIGN.md section 4)"}}
    return out


if __name__ == "__main__":
    sys.exit(main())
