"""Thin numpy-facing wrapper over the C ABI (include/pyrad_b200.h).  Holds no physics."""
import ctypes as C

import numpy as np

from . import _lib

K_BOLTZ = 1.38064852E-23          # pyradClasses.py:16
P0 = 1013.25

OUT_F64, OUT_F32 = 0, 1
K2_GENERAL, K2_CLASSED, K2_FARFIELD = 0, 1, 2
OPT_BATCH_LAYERS, OPT_FUSE_SINGLE_LAYER, OPT_RECORD_BUDGET_MB, OPT_POINT_KERNEL, OPT_FOLD_TMA, OPT_SPLIT_TILES = 1, 2, 3, 4, 5, 6
PEER_HANDLE_BYTES = 64
REFLECTIONS = {"lambertian": 0, "specular": 1}       # PRB_REFLECT_LAMBERTIAN, PRB_REFLECT_SPECULAR


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


class PinnedBlock:
    """A block of page-locked host memory (prb_host_alloc) carved into numpy arrays; freed when the block object and every
    array carved from it are gone (each array's base keeps the block alive).
    `ok` is False when no CUDA device is usable (the arrays are then ordinary numpy arrays)."""

    def __init__(self, nbytes):
        self._lib = _lib.load()
        self.nbytes = int(nbytes)
        self.ptr = self._lib.prb_host_alloc(self.nbytes) if self.nbytes else None
        self.ok = bool(self.ptr)
        self._used = 0

    def array(self, n, dtype=np.float64):
        """The next n elements of the block as a numpy array (64-byte aligned); an ordinary array when not pinned."""
        dt = np.dtype(dtype)
        start = (self._used + 63) & ~63
        if not self.ok or start + n * dt.itemsize > self.nbytes:
            return np.empty(n, dtype=dt)
        self._used = start + n * dt.itemsize
        buf = (C.c_char * (n * dt.itemsize)).from_address(self.ptr + start)
        buf._block = self                    # array -> its ctypes base -> this block: freed with the LAST array, not before
        return np.frombuffer(buf, dtype=dt, count=n)

    def __del__(self):
        try:
            if self.ok and self.ptr:
                self._lib.prb_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


class _Lease:
    """Hands a pooled block back when the array carved from it (and every view of it) is gone."""

    def __init__(self, pool, block):
        self.pool, self.block = pool, block

    def __del__(self):
        try:
            self.pool._give_back(self.block)
        except Exception:
            pass


class ResultPool:
    """Page-locked result arrays that are reused: a spectrum of 3 M doubles copied into a fresh np.empty() pays for 6000
    first-touch page faults and a staged copy (~1.2 ms); into a page-locked array that already exists it is one DMA
    (~0.45 ms).  array() returns an ordinary-looking numpy array backed by a pinned block; when the caller drops it the
    block goes back on the free list (at most `max_free` blocks / `max_bytes` are kept, the rest is released)."""

    def __init__(self, max_free=8, max_bytes=1 << 30):
        self.free = {}
        self.max_free, self.max_bytes = max_free, max_bytes
        self.held = 0

    def array(self, shape, dtype=np.float64):
        dt = np.dtype(dtype)
        n = int(np.prod(shape))
        nbytes = n * dt.itemsize
        if nbytes < (1 << 20):                       # small results: not worth a pinned block
            return np.empty(shape, dtype=dt)
        lst = self.free.get(nbytes)
        if lst:
            block = lst.pop()
            self.held -= nbytes
        else:
            block = PinnedBlock(nbytes)
            if not block.ok:
                return np.empty(shape, dtype=dt)
        buf = (C.c_char * nbytes).from_address(block.ptr)
        buf._lease = _Lease(self, block)
        return np.frombuffer(buf, dtype=dt, count=n).reshape(shape)

    def _give_back(self, block):
        lst = self.free.setdefault(block.nbytes, [])
        if sum(len(v) for v in self.free.values()) < self.max_free and self.held + block.nbytes <= self.max_bytes:
            lst.append(block)
            self.held += block.nbytes

    def clear(self):
        self.free.clear()
        self.held = 0


def window_len(cutoff, res):
    """W = len(np.arange(0, cutoff, res)) (pyradClasses.py:377) -- numpy's own length rule."""
    return len(np.arange(0, cutoff, res))


def grid_len(range_min, range_max, res):
    """N = int((rangeMax - rangeMin) / res) (pyradClasses.py:672, 700)."""
    return int((range_max - range_min) / res)


def number_density_weight(conc, P, T):
    """absCoef factor conc * P / 1E4 / k / T, left to right (pyradClasses.py:583)."""
    return conc * P / 1E4 / K_BOLTZ / T


def flux_boundary_args(emissivity=None, reflection="lambertian", t_top=0.0):
    """Checked arguments of prb_set_flux_boundaries: (table_nu, table_emissivity, reflection code, t_top).

    emissivity: None (a black surface: an empty table), a scalar (a one-entry table: a constant), or a pair (nu, eps) of
    1-d arrays of one length, nu in cm-1 finite and strictly ascending; every emissivity finite and in [0, 1].
    reflection: "lambertian" or "specular"; t_top: the top's temperature in K, finite and >= 0.  ValueError otherwise."""
    if emissivity is None:
        nu, eps = np.zeros(0), np.zeros(0)
    elif np.ndim(emissivity) == 0:
        nu, eps = np.zeros(1), np.array([float(emissivity)])
    else:
        if len(emissivity) != 2:
            raise ValueError("emissivity must be None, a scalar or a pair (nu, eps)")
        nu, eps = _f64(emissivity[0]), _f64(emissivity[1])
        if nu.ndim != 1 or nu.shape != eps.shape or nu.size < 1:
            raise ValueError("emissivity: nu and eps must be 1-d arrays of one length, at least one entry")
        if not np.all(np.isfinite(nu)) or not np.all(np.diff(nu) > 0):
            raise ValueError("emissivity: nu must be finite and strictly ascending")
    if not np.all((eps >= 0) & (eps <= 1)):
        raise ValueError("emissivity must be finite and in [0, 1]")
    if not isinstance(reflection, str) or reflection not in REFLECTIONS:
        raise ValueError("reflection must be one of %s" % sorted(REFLECTIONS))
    t_top = float(t_top)
    if not (np.isfinite(t_top) and t_top >= 0):
        raise ValueError("t_top must be finite and >= 0")
    return nu, eps, REFLECTIONS[reflection], t_top


def solar_source_args(irradiance=None, mu_sun=1.0):
    """Checked arguments of prb_set_solar_source: (table_nu, table_irradiance, mu_sun).

    irradiance: None (no Sun: an empty table) or a pair (nu, S) of 1-d arrays of one length, at least two entries; nu in
    cm-1 finite and strictly ascending, S in W m-2 (cm-1)-1 on a plane normal to the beam, finite and >= 0.  mu_sun: the
    cosine of the solar zenith angle, in (0, 1]; ignored without a Sun.  ValueError otherwise."""
    if irradiance is None:
        return np.zeros(0), np.zeros(0), 1.0
    if not hasattr(irradiance, "__len__") or len(irradiance) != 2:
        raise ValueError("irradiance must be None or a pair (nu, S)")
    nu, s = _f64(irradiance[0]), _f64(irradiance[1])
    if nu.ndim != 1 or nu.shape != s.shape or nu.size < 2:
        raise ValueError("irradiance: nu and S must be 1-d arrays of one length, at least two entries")
    if not np.all(np.isfinite(nu)) or not np.all(np.diff(nu) > 0):
        raise ValueError("irradiance: nu must be finite and strictly ascending")
    if not np.all(np.isfinite(s) & (s >= 0)):
        raise ValueError("irradiance: S must be finite and >= 0")
    mu_sun = float(mu_sun)
    if not (mu_sun > 0 and mu_sun <= 1):
        raise ValueError("mu_sun must lie in (0, 1]")
    return nu, s, mu_sun


CONTINUUM_KEYS = ("nu", "self", "foreign", "texp")


def continuum_args(table=None, mole_fraction=None):
    """Checked arguments of prb_set_continuum: (table_nu, c_self, c_foreign, t_exp, t_ref, p_ref, mole_fraction).

    table: None (no continuum: empty arrays) or a dict in MT_CKD's form with the 1-d arrays "nu" (cm-1, finite and strictly
    ascending, at least two entries), "self" and "foreign" (cm2 molecule-1 (cm-1)-1, finite and >= 0) and "texp" (the
    self coefficient's temperature exponent, finite), all of one length, and optional "t_ref" (K, default 296.0) and
    "p_ref" (hPa, default 1013.0), finite and > 0.  mole_fraction: the continuum gas's mole fraction per layer, a
    non-empty 1-d array with every entry in [0, 1]; ignored without a table.  ValueError otherwise."""
    if table is None:
        z = np.zeros(0)
        return z, z, z, z, 296.0, 1013.0, z
    if not isinstance(table, dict):
        raise ValueError("continuum table must be None or a dict with keys %s" % (CONTINUUM_KEYS,))
    missing = [k for k in CONTINUUM_KEYS if k not in table]
    if missing:
        raise ValueError("continuum table lacks %s" % missing)
    unknown = sorted(set(table) - set(CONTINUUM_KEYS) - {"t_ref", "p_ref"})
    if unknown:
        raise ValueError("continuum table: unknown keys %s" % unknown)
    nu, cs, cf, tx = (_f64(table[k]) for k in CONTINUUM_KEYS)
    if nu.ndim != 1 or nu.size < 2 or not (nu.shape == cs.shape == cf.shape == tx.shape):
        raise ValueError("continuum table: nu, self, foreign and texp must be 1-d arrays of one length, at least two entries")
    if not np.all(np.isfinite(nu)) or not np.all(np.diff(nu) > 0):
        raise ValueError("continuum table: nu must be finite and strictly ascending")
    if not np.all(np.isfinite(cs) & (cs >= 0) & np.isfinite(cf) & (cf >= 0)):
        raise ValueError("continuum table: self and foreign must be finite and >= 0")
    if not np.all(np.isfinite(tx)):
        raise ValueError("continuum table: texp must be finite")
    t_ref, p_ref = float(table.get("t_ref", 296.0)), float(table.get("p_ref", 1013.0))
    if not (np.isfinite(t_ref) and t_ref > 0 and np.isfinite(p_ref) and p_ref > 0):
        raise ValueError("continuum table: t_ref and p_ref must be finite and > 0")
    if mole_fraction is None:
        raise ValueError("a continuum needs the mole fraction of its gas per layer")
    x = _f64(mole_fraction)
    if x.ndim != 1 or x.size < 1:
        raise ValueError("mole_fraction must be a non-empty 1-d array, one entry per layer")
    if not np.all((x >= 0) & (x <= 1)):
        raise ValueError("every mole fraction must be finite and in [0, 1]")
    return nu, cs, cf, tx, t_ref, p_ref, x


class Engine:
    """One engine per process per device (the C ABI's contract)."""

    def __init__(self, device=0):
        self._lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self._lib.prb_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)
        self.n_lines = 0
        self.n_groups = 0
        self.n_chunk = 0

    # -- lifecycle
    def close(self):
        if getattr(self, "_h", None):
            self._lib.prb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def stream(self):
        """Raw cudaStream_t of the engine (wrap with torch.cuda.ExternalStream for CUDA events)."""
        return int(self._lib.prb_stream(self._h) or 0)

    def synchronize(self):
        _lib.check(self._lib.prb_synchronize(self._h))

    def device_info(self):
        sm, ma, mi, khz = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        fr, to = C.c_size_t(), C.c_size_t()
        _lib.check(self._lib.prb_device_info(self._h, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(khz),
                                             C.byref(fr), C.byref(to)))
        return {"sm_count": sm.value, "cc": (ma.value, mi.value), "sm_clock_khz": khz.value,
                "free_bytes": fr.value, "total_bytes": to.value}

    def measure_peaks(self):
        """Roofline denominators measured on this device: FP32 lane-FMA/s (packed FFMA2 and scalar FFMA streams) and the
        float4 copy bandwidth in bytes/s (read + write)."""
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        _lib.check(self._lib.prb_measure_peaks(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return {"ffma2_lane_fma_per_s": a.value, "ffma_lane_fma_per_s": b.value, "copy_bytes_per_s": c.value}

    def set_k2_variant(self, variant=K2_CLASSED, points_per_thread=0):
        _lib.check(self._lib.prb_set_k2_variant(self._h, int(variant), int(points_per_thread)))

    def set_option(self, option, value):
        _lib.check(self._lib.prb_set_option(self._h, int(option), int(value)))

    def set_narrow_threshold(self, wm_below=-1):
        _lib.check(self._lib.prb_set_narrow_threshold(self._h, int(wm_below)))

    # -- data
    def upload_lines(self, lines, n_groups=1):
        """lines: dict with nu, sw, gamma_air, gamma_self, elower, n_air, delta_air (+ optional int32 group),
        ascending in nu."""
        cols = [_f64(lines[k]) for k in ("nu", "sw", "gamma_air", "gamma_self", "elower", "n_air", "delta_air")]
        n = cols[0].size
        grp = lines.get("group") if hasattr(lines, "get") else None
        gp = None
        if grp is not None:
            grp = np.ascontiguousarray(grp, dtype=np.int32)
            gp = grp.ctypes.data_as(C.POINTER(C.c_int32))
        _lib.check(self._lib.prb_upload_lines(self._h, n, *[_dp(c) for c in cols], gp, int(n_groups)))
        self.n_lines = n
        self.n_groups = int(n_groups)

    def upload_line_groups(self, groups):
        """groups: one dict of SoA columns per isotopologue, each ascending in nu -- uploaded from where they are (a table
        of column pointers per group: no merge, no concatenation); line_sum_groups() then returns one row per group from
        one prepass + one line-sum launch."""
        names = ("nu", "sw", "gamma_air", "gamma_self", "elower", "n_air", "delta_air")
        G = len(groups)
        keep = [[_f64(g[k]) for g in groups] for k in names]
        counts = np.array([c.size for c in keep[0]], dtype=np.int64)
        tables = [(C.POINTER(C.c_double) * G)(*[_dp(c) for c in col]) for col in keep]
        _lib.check(self._lib.prb_upload_line_groups(self._h, G, counts.ctypes.data_as(C.POINTER(C.c_int64)), *tables))
        self.n_lines = int(counts.sum())
        self.n_groups = G

    def ingest_csv(self, text, wave_min, wave_max):
        """HITRAN-online CSV bytes -> the engine's line list, parsed on the device (K5).  Returns the line count."""
        blob = bytes(text)
        n = C.c_int64()
        _lib.check(self._lib.prb_ingest_hitran_csv(self._h, blob, len(blob), float(wave_min), float(wave_max),
                                                   C.byref(n)))
        self.n_lines = n.value
        self.n_groups = 1
        return n.value

    def download_lines(self):
        """The device-resident line list as SoA float64 columns (hitran_io.LINE_COLUMNS)."""
        n = int(self._lib.prb_line_count(self._h))
        if n < 0:
            raise _lib.EngineError(-3, "no line list on the device")
        names = ("nu", "sw", "a", "elower", "gamma_air", "gamma_self", "delta_air", "n_air")
        cols = {k: np.empty(n) for k in names}
        _lib.check(self._lib.prb_download_lines(self._h, *[_dp(cols[k]) for k in names]))
        return cols

    def parse_xsc_text(self, text):
        """Two-column xsc table bytes -> (wavenumber, cross section) float64 arrays, parsed on the device (K5)."""
        blob = bytes(text)
        cap = blob.count(b"\n") + 1
        wn, xs = np.empty(cap), np.empty(cap)
        n = C.c_int64()
        _lib.check(self._lib.prb_parse_xsc_text(self._h, blob, len(blob), cap, _dp(wn), _dp(xs), C.byref(n)))
        return wn[:n.value].copy(), xs[:n.value].copy()

    def set_grid(self, range_min, res, n_total, i_begin=0, i_end=None):
        i_end = n_total if i_end is None else i_end
        _lib.check(self._lib.prb_set_grid(self._h, float(range_min), float(res), int(n_total), int(i_begin),
                                          int(i_end)))
        self.n_chunk = int(i_end) - int(i_begin)
        self.n_total = int(n_total)
        self.i_begin, self.i_end = int(i_begin), int(i_end)
        self._res = float(res)
        self.range_min = float(range_min)

    # -- kernels
    def layer_prepass(self, T, P, conc, molmass, q_t, q_296, window, weight=None):
        g = self.n_groups
        arrs = [_f64(np.broadcast_to(np.asarray(a, dtype=np.float64), (g,))) for a in (conc, molmass, q_t, q_296)]
        w = _f64(np.broadcast_to(np.asarray(weight, dtype=np.float64), (g,))) if weight is not None else None
        _lib.check(self._lib.prb_layer_prepass(self._h, float(T), float(P), g, *[_dp(a) for a in arrs], _dp(w),
                                               int(window)))

    def line_sum(self):
        out = np.empty(self.n_chunk, dtype=np.float64)
        _lib.check(self._lib.prb_line_sum(self._h, _dp(out)))
        return out

    def _result(self, shape):
        """A result array: from the page-locked pool when one is attached (Engine.result_pool), else np.empty."""
        pool = getattr(self, "result_pool", None)
        return pool.array(shape) if pool is not None else np.empty(shape, dtype=np.float64)

    def line_sum_groups(self, to_host=True):
        """One row per group (prb_line_sum_groups); to_host=False leaves them on the device for layer_spectra_resident()."""
        # (fetched once per layer state and cached by the caller: an ordinary array, not a pooled page-locked one)
        out = np.empty((self.n_groups, self.n_chunk), dtype=np.float64) if to_host else None
        _lib.check(self._lib.prb_line_sum_groups(self._h, _dp(out)))
        return out

    def layer_spectra_resident(self, group_weight, depth_cm, t_layer, range_max, xsc_weight=None, radiance_in=None,
                               want=("abs_coef", "transmittance", "radiance")):
        """k, T, Layer.transmission from the device-resident per-group rows (+ resident xsc tables): one D2H per output."""
        w = _f64(group_weight)
        xw = _f64(xsc_weight) if xsc_weight is not None and len(xsc_weight) else None
        rin = _f64(radiance_in) if radiance_in is not None else None
        n = self.n_chunk
        k = self._result(n) if "abs_coef" in want else None
        t = self._result(n) if "transmittance" in want else None
        r = self._result(n) if ("radiance" in want and rin is not None) else None
        _lib.check(self._lib.prb_layer_spectra_resident(self._h, _dp(w), _dp(xw), float(depth_cm), float(t_layer),
                                                        float(range_max), _dp(rin), _dp(k), _dp(t), _dp(r)))
        return k, t, r

    def line_sum_dev(self, dev_ptr, out_mode=OUT_F64):
        _lib.check(self._lib.prb_line_sum_dev(self._h, C.c_void_p(int(dev_ptr)), int(out_mode)))

    def pair_count(self):
        n = self._lib.prb_pair_count(self._h)
        if n < 0:
            raise _lib.EngineError(int(n), _lib.last_error())
        return int(n)

    def debug_line_params(self):
        n = self.n_lines
        out = {k: np.empty(n, dtype=np.float64) for k in ("nu_shift", "gamma_l", "gamma_d", "s_t")}
        reg = np.empty(n, dtype=np.int32)
        idx = np.empty(n, dtype=np.int64)
        _lib.check(self._lib.prb_debug_line_params(
            self._h, _dp(out["nu_shift"]), _dp(out["gamma_l"]), _dp(out["gamma_d"]), _dp(out["s_t"]),
            reg.ctypes.data_as(C.POINTER(C.c_int32)), idx.ctypes.data_as(C.POINTER(C.c_int64))))
        out["regime"] = reg
        out["index"] = idx
        return out

    def cross_section(self, T, P, conc, molmass, q_t, q_296, cutoff, res=None, weight=None):
        """prepass + line sum on the current grid: Isotope.createCrossSection (pyradClasses.py:361-400)."""
        res = self._res if res is None else res
        self.layer_prepass(T, P, conc, molmass, q_t, q_296, window_len(cutoff, res), weight)
        return self.line_sum()

    def layer_stream(self, sigma, weight, depth_cm, t_layer, axis, radiance_in=None,
                     want=("abs_coef", "transmittance", "radiance")):
        """axis = (x0, dx, x_last, n) of the np.linspace grid (Layer.xAxis)."""
        sigma = _f64(np.atleast_2d(sigma))
        n_mol, n = sigma.shape
        x0, dx, x_last, n_axis = axis
        assert n_axis == n
        w = _f64(weight)
        rin = _f64(radiance_in) if radiance_in is not None else None
        k = np.empty(n) if "abs_coef" in want else None
        t = np.empty(n) if "transmittance" in want else None
        r = np.empty(n) if ("radiance" in want and rin is not None) else None
        _lib.check(self._lib.prb_layer_stream(self._h, n, n_mol, _dp(sigma), _dp(w), float(depth_cm), float(t_layer),
                                              float(x0), float(dx), float(x_last), _dp(rin), _dp(k), _dp(t), _dp(r)))
        return k, t, r

    def planck(self, axis, temp):
        x0, dx, x_last, n = axis
        out = np.empty(n)
        _lib.check(self._lib.prb_planck(self._h, n, float(x0), float(dx), float(x_last), float(temp), _dp(out)))
        return out

    def xsc_place(self, n_out, dst0, src0, count, file_x, file_y, interp, ax0=0.0, adelta=0.0):
        fy = _f64(file_y)
        fx = _f64(file_x) if file_x is not None else None
        out = np.empty(n_out)
        _lib.check(self._lib.prb_xsc_place(self._h, n_out, int(dst0), int(src0), int(count), int(bool(interp)),
                                           float(ax0), float(adelta), fy.size, _dp(fx), _dp(fy), _dp(out)))
        return out

    def xsc_resident(self, slot, n_out, dst0, src0, count, file_x, file_y, interp, ax0=0.0, adelta=0.0):
        """Keep xsc table `slot` on the device with its placement plan (the arguments of xsc_place); the following
        atmosphere() / gas_cell_host() calls add it to every layer's k(nu) with the mole fractions of set_xsc_conc()."""
        fy = _f64(file_y)
        fx = _f64(file_x) if file_x is not None else None
        _lib.check(self._lib.prb_xsc_resident(self._h, int(slot), int(n_out), int(dst0), int(src0), int(count),
                                              int(bool(interp)), float(ax0), float(adelta), fy.size, _dp(fx), _dp(fy)))

    def set_layer_line_range(self, nu_lo=None, nu_hi=None):
        """Per-layer open intervals (nu_lo[l], nu_hi[l]) of the line wavenumbers that take part in layer l of the following
        atmosphere() calls -- the reference's gatherData(effectiveRangeMin, effectiveRangeMax) filter when ONE line list
        serves a column of layers with different cutoffs; no arguments: every line takes part again."""
        if nu_lo is None:
            _lib.check(self._lib.prb_set_layer_line_range(self._h, 0, None, None))
            return
        lo, hi = _f64(nu_lo), _f64(nu_hi)
        if lo.shape != hi.shape or lo.ndim != 1:
            raise ValueError("set_layer_line_range: nu_lo and nu_hi must be 1-d arrays of one length")
        _lib.check(self._lib.prb_set_layer_line_range(self._h, lo.size, _dp(lo), _dp(hi)))

    def set_xsc_conc(self, conc):
        """conc: (L, n_xsc) mole fractions of the resident xsc tables in every layer of the next atmosphere() call."""
        c = _f64(np.atleast_2d(conc))
        _lib.check(self._lib.prb_set_xsc_conc(self._h, c.shape[0], c.shape[1], _dp(c)))

    def xsc_clear(self):
        _lib.check(self._lib.prb_xsc_clear(self._h))

    def set_continuum(self, table=None, mole_fraction=None):
        """A water-vapour continuum in MT_CKD's form for every later atmosphere() / gas cell with len(mole_fraction)
        layers (prb_set_continuum; arguments as continuum_args).  Row l of the k matrix gains, before the fold,
        n_l rho_l R(nu, T_l) [x_l (t_ref/T_l)^texp C_self + (1 - x_l) C_foreign], the table interpolated onto the grid
        (0 outside it for the coefficients).  The table must suit the line shape: MT_CKD's belongs to lines cut at
        25 cm-1 with the 25 cm-1 value subtracted, this path cuts at 5 P/p0 cm-1.  No arguments: no continuum again."""
        nu, cs, cf, tx, t_ref, p_ref, x = continuum_args(table, mole_fraction)
        if not nu.size:
            _lib.check(self._lib.prb_set_continuum(self._h, 0, None, None, None, None, t_ref, p_ref, 0, None))
            return
        _lib.check(self._lib.prb_set_continuum(self._h, nu.size, _dp(nu), _dp(cs), _dp(cf), _dp(tx), t_ref, p_ref,
                                               x.size, _dp(x)))

    def atmosphere_call(self, depth_cm, t_layer, p_layer, conc, molmass, q_t, q_296, window, t_surface, range_max):
        """The prb_atmosphere call with its arguments marshalled ONCE: returns a zero-argument callable for callers that
        repeat the same column (a step loop) -- per call only the ctypes transition is left on the host."""
        L = len(t_layer)
        g = self.n_groups
        keep = [_f64(np.broadcast_to(np.asarray(depth_cm, dtype=np.float64), (L,))), _f64(t_layer), _f64(p_layer),
                _f64(np.broadcast_to(np.asarray(conc, dtype=np.float64), (L, g))),
                _f64(np.broadcast_to(np.asarray(molmass, dtype=np.float64), (g,))),
                _f64(np.broadcast_to(np.asarray(q_t, dtype=np.float64), (L, g))),
                _f64(np.broadcast_to(np.asarray(q_296, dtype=np.float64), (g,)))]
        win = np.ascontiguousarray(window, dtype=np.int64)
        ptrs = [_dp(a) for a in keep] + [win.ctypes.data_as(C.POINTER(C.c_int64))]
        fn, h, ts, rm = self._lib.prb_atmosphere, self._h, float(t_surface), float(range_max)

        def call():
            rc = fn(h, L, g, *ptrs, ts, rm)
            if rc:
                _lib.check(rc)
            self.atm_layers = L
        call.keepalive = (keep, win)
        return call

    def atmosphere(self, depth_cm, t_layer, p_layer, conc, molmass, q_t, q_296, window, t_surface, range_max):
        """conc, q_t: (L, G); molmass, q_296: (G,).  Runs K1+K2 per layer and the K3 fold on the device."""
        self.atmosphere_call(depth_cm, t_layer, p_layer, conc, molmass, q_t, q_296, window, t_surface, range_max)()

    def gas_cell_host_call(self, lines, n_groups, range_min, res, n_total, i_begin, i_end, depth_cm, T, P, conc, molmass,
                           q_t, q_296, window, t_surface, range_max):
        """prb_gas_cell_host with its arguments marshalled once (see atmosphere_call); the line columns are read from
        the given host arrays on every call."""
        cols = [_f64(lines[k]) for k in ("nu", "sw", "gamma_air", "gamma_self", "elower", "n_air", "delta_air")]
        n = cols[0].size
        grp = lines.get("group") if hasattr(lines, "get") else None
        gp = None
        if grp is not None:
            grp = np.ascontiguousarray(grp, dtype=np.int32)
            gp = grp.ctypes.data_as(C.POINTER(C.c_int32))
        g = int(n_groups)
        arrs = [_f64(np.broadcast_to(np.asarray(a, dtype=np.float64), (g,))) for a in (conc, molmass, q_t, q_296)]
        args = ([self._h, n] + [_dp(c) for c in cols] + [gp, g, float(range_min), float(res), int(n_total), int(i_begin),
                int(i_end), float(depth_cm), float(T), float(P)] + [_dp(a) for a in arrs] +
                [int(window), float(t_surface), float(range_max)])
        fn = self._lib.prb_gas_cell_host

        def call():
            rc = fn(*args)
            if rc:
                _lib.check(rc)
            self.n_lines, self.n_groups = n, g
            self.atm_layers = 1
            self.n_chunk = int(i_end) - int(i_begin)
            self.n_total = int(n_total)
            self.i_begin, self.i_end = int(i_begin), int(i_end)
            self._res = float(res)
            self.range_min = float(range_min)
        call.keepalive = (cols, grp, arrs)
        return call

    def gas_cell_host(self, lines, n_groups, range_min, res, n_total, i_begin, i_end, depth_cm, T, P, conc, molmass,
                      q_t, q_296, window, t_surface, range_max):
        """upload_lines + set_grid + atmosphere(one layer) in ONE call with the host->device copies overlapped with
        the compute (prb_gas_cell_host).  Results: atmosphere_read*(), or the buffers given to set_result_host()."""
        self.gas_cell_host_call(lines, n_groups, range_min, res, n_total, i_begin, i_end, depth_cm, T, P, conc, molmass,
                                q_t, q_296, window, t_surface, range_max)()

    def atmosphere_read(self):
        rad = np.empty(self.n_chunk)
        tr = np.empty(self.n_chunk)
        _lib.check(self._lib.prb_atmosphere_read(self._h, _dp(rad), _dp(tr)))
        return rad, tr

    def atmosphere_read_f32(self, rad=None, tr=None):
        """Copy the FP32 device results into caller-owned float32 host arrays (pinned or not), no widening."""
        fp = C.POINTER(C.c_float)
        _lib.check(self._lib.prb_atmosphere_read_f32(
            self._h, rad.ctypes.data_as(fp) if rad is not None else None,
            tr.ctypes.data_as(fp) if tr is not None else None))

    def atmosphere_fluxes(self, mu, weights, rows=False):
        """Hemispheric fluxes of the last column (prb_atmosphere_fluxes) for the angular quadrature (mu, weights), 1 to 4
        nodes: (flux_up, flux_down), float64 W m-2 per level (L+1: level 0 = surface, L = top; this chunk's share).  With
        rows=True also (rad_up_top, rad_down_surface), float32 (n_mu, chunk): the radiance leaving the top and reaching
        the surface along every mu."""
        m, w = _f64(np.atleast_1d(mu)), _f64(np.atleast_1d(weights))
        if m.ndim != 1 or m.shape != w.shape:
            raise ValueError("atmosphere_fluxes: mu and weights must be 1-d arrays of one length")
        L = int(getattr(self, "atm_layers", 0))
        up, down = np.zeros(L + 1), np.zeros(L + 1)
        fp = C.POINTER(C.c_float)
        ru = np.empty((m.size, self.n_chunk), dtype=np.float32) if rows else None
        rd = np.empty((m.size, self.n_chunk), dtype=np.float32) if rows else None
        _lib.check(self._lib.prb_atmosphere_fluxes(self._h, m.size, _dp(m), _dp(w), _dp(up) if L else None,
                                                   _dp(down) if L else None, ru.ctypes.data_as(fp) if rows else None,
                                                   rd.ctypes.data_as(fp) if rows else None))
        return (up, down, ru, rd) if rows else (up, down)

    def atmosphere_band_fluxes(self, mu, weights, edges):
        """Band fluxes of the last column (prb_atmosphere_band_fluxes): the fluxes of atmosphere_fluxes split by the
        wavenumber bands edges[b] <= nu < edges[b+1] (cm-1, strictly ascending; nu the column's linspace axis).  Returns
        (band_up, band_down), float64 W m-2 of shape (n_bands, L+1): level 0 = surface, L = top; this chunk's share."""
        m, w, ed = _f64(np.atleast_1d(mu)), _f64(np.atleast_1d(weights)), _f64(np.atleast_1d(edges))
        if m.ndim != 1 or m.shape != w.shape:
            raise ValueError("atmosphere_band_fluxes: mu and weights must be 1-d arrays of one length")
        if ed.ndim != 1:
            raise ValueError("atmosphere_band_fluxes: edges must be a 1-d array")
        L = int(getattr(self, "atm_layers", 0))
        nb = max(ed.size - 1, 0)
        up, down = np.zeros((nb, L + 1)), np.zeros((nb, L + 1))
        _lib.check(self._lib.prb_atmosphere_band_fluxes(self._h, m.size, _dp(m), _dp(w), ed.size - 1, _dp(ed),
                                                        _dp(up) if up.size else None, _dp(down) if down.size else None))
        return up, down

    def set_flux_boundaries(self, emissivity=None, reflection="lambertian", t_top=0.0):
        """The surface and top boundaries of every later atmosphere_fluxes / atmosphere_band_fluxes call
        (prb_set_flux_boundaries; arguments as flux_boundary_args).  The surface emits eps(nu) B(nu, T_surface) and
        reflects 1 - eps(nu) of the sky's radiance, diffusely (Lambertian) or along the same mu (specular); eps is
        np.interp over the table on the column's grid.  The top sends B(nu, t_top) down.  No arguments: a black surface
        and nothing from the top again.  The column's own radiance (atmosphere_read) is not affected."""
        nu, eps, refl, t_top = flux_boundary_args(emissivity, reflection, t_top)
        _lib.check(self._lib.prb_set_flux_boundaries(self._h, nu.size, _dp(nu) if nu.size else None,
                                                     _dp(eps) if eps.size else None, refl, t_top))

    def set_solar_source(self, irradiance=None, mu_sun=1.0):
        """The Sun of every later atmosphere_fluxes / atmosphere_band_fluxes call (prb_set_solar_source; arguments as
        solar_source_args): a beam along mu_sun with irradiance S(nu) at the top, np.interp over the table on the
        column's grid and 0 outside it, absorbed on its way down and reflected by the surface of set_flux_boundaries
        (1 - eps of it, as that call's reflection says).  flux_down includes the beam, and flux_up its reflection.  No
        arguments: no Sun again.  The column's own radiance (atmosphere_read) is not affected."""
        nu, s, mu_sun = solar_source_args(irradiance, mu_sun)
        _lib.check(self._lib.prb_set_solar_source(self._h, nu.size, _dp(nu) if nu.size else None,
                                                  _dp(s) if s.size else None, mu_sun))

    def set_result_host(self, rad=None, tr=None):
        """Register pinned float32 host arrays that every following atmosphere() fills directly from the device
        kernels (zero-copy); call with no arguments to switch it off."""
        fp = C.POINTER(C.c_float)
        if rad is None and tr is None:
            _lib.check(self._lib.prb_set_result_host(self._h, None, None, 0))
            return
        assert rad.dtype == np.float32 and tr.dtype == np.float32 and rad.size == tr.size
        _lib.check(self._lib.prb_set_result_host(self._h, rad.ctypes.data_as(fp), tr.ctypes.data_as(fp), rad.size))

    def set_timing(self, enabled=True):
        _lib.check(self._lib.prb_set_timing(self._h, int(bool(enabled))))

    def atmosphere_timing(self):
        a, b, c = C.c_float(), C.c_float(), C.c_float()
        _lib.check(self._lib.prb_atmosphere_timing(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return {"k1_ms": a.value, "k2_ms": b.value, "k3_ms": c.value}

    def atmosphere_layer_timing(self, n_layers):
        a = np.zeros(n_layers, dtype=np.float32)
        b = np.zeros(n_layers, dtype=np.float32)
        fp = C.POINTER(C.c_float)
        _lib.check(self._lib.prb_atmosphere_layer_timing(self._h, int(n_layers), a.ctypes.data_as(fp), b.ctypes.data_as(fp)))
        return a, b

    def atmosphere_result_dev(self):
        a, b = C.c_void_p(), C.c_void_p()
        _lib.check(self._lib.prb_atmosphere_result_dev(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    # -- section 8(f) rows: survey, integrals, derived spectra
    def line_survey(self, n_out):
        """Isotope.createLineSurvey (pyradClasses.py:409-428) of the uploaded lines on the current grid."""
        out = np.empty(int(n_out))
        _lib.check(self._lib.prb_line_survey(self._h, int(n_out), _dp(out)))
        return out

    def integrate_spectrum(self, spectrum, unit_angle, res):
        """integrateSpectrum (pyradClasses.py:26-29)."""
        x = _f64(spectrum)
        v = C.c_double()
        _lib.check(self._lib.prb_integrate_spectrum(self._h, x.size, _dp(x), float(unit_angle), float(res), C.byref(v)))
        return v.value

    def atmosphere_integrate(self, unit_angle, res):
        """(integral of the device-resident radiance, sum of the total transmittance) over the owned chunk."""
        a, b = C.c_double(), C.c_double()
        _lib.check(self._lib.prb_atmosphere_integrate(self._h, float(unit_angle), float(res), C.byref(a), C.byref(b)))
        return a.value, b.value

    def derived_spectra(self, transmittance, want=("emissivity", "optical_depth", "absorbance")):
        t = _f64(transmittance)
        out = {k: (np.empty(t.size) if k in want else None) for k in ("emissivity", "optical_depth", "absorbance")}
        _lib.check(self._lib.prb_derived_spectra(self._h, t.size, _dp(t), _dp(out["emissivity"]),
                                                 _dp(out["optical_depth"]), _dp(out["absorbance"])))
        return out

    def atmosphere_launches(self):
        """Kernels launched by the last atmosphere() call."""
        return int(self._lib.prb_atmosphere_launches(self._h))

    # -- multi-GPU: peer-memory gather of the finished spectra (include/pyrad_b200.h, "multi-GPU")
    def peer_alloc(self, rank, world, max_chunk_points):
        """Allocate this rank's gather buffer; returns its 64-byte CUDA IPC handle (bytes)."""
        buf = C.create_string_buffer(PEER_HANDLE_BYTES)
        _lib.check(self._lib.prb_peer_alloc(self._h, int(rank), int(world), int(max_chunk_points), buf))
        self._peer_world = int(world)
        return buf.raw

    def peer_connect(self, handles):
        """handles: the world handles in rank order (list of bytes or one bytes object)."""
        blob = b"".join(handles) if not isinstance(handles, (bytes, bytearray)) else bytes(handles)
        buf = C.create_string_buffer(blob, len(blob))
        _lib.check(self._lib.prb_peer_connect(self._h, buf))

    def peer_disconnect(self):
        _lib.check(self._lib.prb_peer_disconnect(self._h))

    def peer_gathered_dev(self):
        """(radiance_ptr, transmittance_ptr, ld): float[world][ld] arrays of the last step on this device."""
        a, b, ld = C.c_void_p(), C.c_void_p(), C.c_int64()
        _lib.check(self._lib.prb_peer_gathered_dev(self._h, C.byref(a), C.byref(b), C.byref(ld)))
        return a.value, b.value, ld.value

    def atmosphere_kmatrix_dev(self):
        p, ld = C.c_void_p(), C.c_int64()
        _lib.check(self._lib.prb_atmosphere_kmatrix_dev(self._h, C.byref(p), C.byref(ld)))
        return p.value, ld.value


def linspace_axis(range_min, range_max, n):
    """(x0, dx, x_last, n) reproducing np.linspace(range_min, range_max, n, endpoint=True) bit for bit:
    numpy forms arange(n) * step + start and overwrites the last sample with stop (Layer.xAxis,
    pyradClasses.py:703-705)."""
    n = int(n)
    step = (range_max - range_min) / (n - 1) if n > 1 else 0.0
    return float(range_min), float(step), float(range_max), n
