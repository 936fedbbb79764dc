"""ctypes binding of libpyrad_b200.so -- the only way Python reaches the CUDA engine.

The prototypes below are exactly the declarations in ``include/pyrad_b200.h``.  There is no
CPU fallback anywhere in this package: if the shared library is missing, or no B200-class
device is present, calls raise ``EngineUnavailable`` loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PRB_LIB") or os.path.join(_HERE, "libpyrad_b200.so")   # PRB_LIB: development A/B builds only


class EngineUnavailable(RuntimeError):
    pass


class EngineError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libpyrad_b200 error %d: %s" % (code, msg))
        self.code = code


_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_lp = C.POINTER(C.c_int64)
_vp = C.c_void_p
_i64 = C.c_int64
_i32 = C.c_int32
_d = C.c_double

#: symbol -> (restype, argtypes); mirrors include/pyrad_b200.h one to one
PROTOTYPES = {
    "prb_abi_version": (C.c_int, []),
    "prb_last_error": (C.c_char_p, []),
    "prb_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "prb_destroy": (C.c_int, [_vp]),
    "prb_stream": (_vp, [_vp]),
    "prb_synchronize": (C.c_int, [_vp]),
    "prb_host_alloc": (_vp, [C.c_size_t]),
    "prb_host_free": (C.c_int, [_vp]),
    "prb_device_info": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                  C.POINTER(C.c_int), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "prb_measure_peaks": (C.c_int, [_vp, _dp, _dp, _dp]),
    "prb_set_k2_variant": (C.c_int, [_vp, C.c_int, C.c_int]),
    "prb_set_narrow_threshold": (C.c_int, [_vp, _i64]),
    "prb_upload_lines": (C.c_int, [_vp, _i64, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _ip, _i32]),
    "prb_upload_line_groups": (C.c_int, [_vp, _i32, _lp] + [C.POINTER(_dp)] * 7),
    "prb_ingest_hitran_csv": (C.c_int, [_vp, C.c_char_p, _i64, _d, _d, _lp]),
    "prb_download_lines": (C.c_int, [_vp, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp]),
    "prb_line_count": (_i64, [_vp]),
    "prb_parse_xsc_text": (C.c_int, [_vp, C.c_char_p, _i64, _i64, _dp, _dp, _lp]),
    "prb_debug_parse_double": (C.c_int, [C.c_char_p, _i64, _dp]),
    "prb_set_grid": (C.c_int, [_vp, _d, _d, _i64, _i64, _i64]),
    "prb_layer_prepass": (C.c_int, [_vp, _d, _d, _i32, _dp, _dp, _dp, _dp, _dp, _i64]),
    "prb_line_sum": (C.c_int, [_vp, _dp]),
    "prb_line_sum_dev": (C.c_int, [_vp, _vp, C.c_int]),
    "prb_line_sum_groups": (C.c_int, [_vp, _dp]),
    "prb_layer_spectra_resident": (C.c_int, [_vp, _dp, _dp, _d, _d, _d, _dp, _dp, _dp, _dp]),
    "prb_pair_count": (_i64, [_vp]),
    "prb_debug_line_params": (C.c_int, [_vp, _dp, _dp, _dp, _dp, _ip, _lp]),
    "prb_layer_stream": (C.c_int, [_vp, _i64, _i32, _dp, _dp, _d, _d, _d, _d, _d, _dp, _dp, _dp, _dp]),
    "prb_planck": (C.c_int, [_vp, _i64, _d, _d, _d, _d, _dp]),
    "prb_xsc_place": (C.c_int, [_vp, _i64, _i64, _i64, _i64, C.c_int, _d, _d, _i64, _dp, _dp, _dp]),
    "prb_xsc_resident": (C.c_int, [_vp, _i32, _i64, _i64, _i64, _i64, C.c_int, _d, _d, _i64, _dp, _dp]),
    "prb_set_xsc_conc": (C.c_int, [_vp, _i32, _i32, _dp]),
    "prb_set_continuum": (C.c_int, [_vp, _i64, _dp, _dp, _dp, _dp, _d, _d, _i32, _dp]),
    "prb_set_layer_line_range": (C.c_int, [_vp, _i32, _dp, _dp]),
    "prb_xsc_clear": (C.c_int, [_vp]),
    "prb_atmosphere": (C.c_int, [_vp, _i32, _i32, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _lp, _d, _d]),
    "prb_gas_cell_host": (C.c_int, [_vp, _i64, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _ip, _i32, _d, _d, _i64, _i64, _i64,
                                    _d, _d, _d, _dp, _dp, _dp, _dp, _i64, _d, _d]),
    "prb_atmosphere_result_dev": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp)]),
    "prb_atmosphere_read": (C.c_int, [_vp, _dp, _dp]),
    "prb_atmosphere_read_f32": (C.c_int, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "prb_set_result_host": (C.c_int, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_float), _i64]),
    "prb_set_timing": (C.c_int, [_vp, C.c_int]),
    "prb_atmosphere_timing": (C.c_int, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "prb_atmosphere_layer_timing": (C.c_int, [_vp, _i32, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "prb_atmosphere_kmatrix_dev": (C.c_int, [_vp, C.POINTER(_vp), _lp]),
    "prb_atmosphere_launches": (C.c_int, [_vp]),
    "prb_atmosphere_fluxes": (C.c_int, [_vp, _i32, _dp, _dp, _dp, _dp, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "prb_atmosphere_band_fluxes": (C.c_int, [_vp, _i32, _dp, _dp, _i32, _dp, _dp, _dp]),
    "prb_atmosphere_save_base": (C.c_int, [_vp]),
    "prb_atmosphere_layer_kernels": (C.c_int, [_vp, _i32, _dp, _dp, _i32, _dp, _dp, _dp]),
    "prb_set_flux_boundaries": (C.c_int, [_vp, _i64, _dp, _dp, _i32, _d]),
    "prb_set_solar_source": (C.c_int, [_vp, _i64, _dp, _dp, _d]),
    "prb_set_option": (C.c_int, [_vp, C.c_int, _i64]),
    "prb_line_survey": (C.c_int, [_vp, _i64, _dp]),
    "prb_integrate_spectrum": (C.c_int, [_vp, _i64, _dp, _d, _d, _dp]),
    "prb_atmosphere_integrate": (C.c_int, [_vp, _d, _d, _dp, _dp]),
    "prb_derived_spectra": (C.c_int, [_vp, _i64, _dp, _dp, _dp, _dp]),
    "prb_peer_alloc": (C.c_int, [_vp, C.c_int, C.c_int, _i64, _vp]),
    "prb_peer_connect": (C.c_int, [_vp, _vp]),
    "prb_peer_disconnect": (C.c_int, [_vp]),
    "prb_peer_gathered_dev": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), _lp]),
}

_lib = None


def load():
    """dlopen the in-tree shared library and attach prototypes.  Loading needs no GPU."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise EngineUnavailable(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(pyrad_b200 has no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError here means header and library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().prb_last_error().decode("utf-8", "replace")


def check(rc):
    if rc != 0:
        msg = last_error()
        if rc == -5:
            raise EngineUnavailable(msg)
        raise EngineError(rc, msg)
