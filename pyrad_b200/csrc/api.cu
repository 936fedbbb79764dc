// api.cu -- the C ABI of libpyrad_b200.so (see include/pyrad_b200.h).  Host-side orchestration only:
// buffers, launches, copies.  No physics is evaluated on the CPU and there is no CPU fallback.
#include "../../include/pyrad_b200.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

#include "common.cuh"
#include "k1_prepass.cuh"
#include "k2_line_sum.cuh"
#include "k2_narrow.cuh"
#include "k2_point.cuh"
#include "k3_stream.cuh"
#include "k4_derived.cuh"
#include "k5_ingest.cuh"
#include "k9_peaks.cuh"
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

using namespace prb;

static thread_local std::string g_err = "";

static int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}

#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            char b_[512];                                                                     \
            snprintf(b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),   \
                     __FILE__, __LINE__);                                                     \
            return fail(PRB_ERR_CUDA, b_);                                                    \
        }                                                                                     \
    } while (0)

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    cudaError_t ensure(size_t count) {
        if (count <= n && p) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) n = count;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
};

// Host-side description of one layer of a launch sequence (one K1 table row + one K2 table row).
struct LayerJob {
    double T = 0, P = 0, scale = 1;
    int64_t W = 0, wm = 0, l0 = 0, l1 = 0;   // window, K2 line range [l0, l1)
    int narrow = 0;              // record layout / kernel: 1 = k2_narrow (thread-per-point gather)
    int ppt = 8;                 // points per thread of k2_line_sum for this window
    int slot = 0;                // which slice of the record arrays holds this layer
    const GroupParams *gp_dev = nullptr;
    const double *scale_dev = nullptr;   // pipelined upload: the scale is computed on the device
    DevState *st_dev = nullptr;
    void *out_dev = nullptr;
    bool valid = false;
    double xsc_w[K2_MAX_XSC] = {};   // absCoef weights of the resident xsc tables in this layer (0: none)
    bool filter = false;             // only lines with nu_lo < nu0 < nu_hi take part (prb_set_layer_line_range)
    double nu_lo = 0, nu_hi = 0;
};

// A resident xsc cross-section table (prb_xsc_resident): the file's samples and its placement plan.
struct XscTable {
    int64_t n_out = 0, dst0 = 0, src0 = 0, count = 0, n_file = 0;
    int interp = 0;
    double ax0 = 0, adelta = 0;
    DevBuf<double> fx, fy;
};

// Peer-memory gather buffers (multi-GPU, one process per GPU on one NVLink/NVSwitch node).
struct PeerState {
    int rank = 0, world = 0;
    int64_t ld = 0;                          // floats per rank slot
    unsigned char *local = nullptr;          // this rank's allocation (exported over CUDA IPC)
    unsigned char *base[K2_MAX_PEERS] = {};  // every rank's allocation as mapped here (base[rank] == local)
    bool connected = false;
    unsigned int epoch = 0;                  // collective step counter (all ranks advance together)
    size_t bytes = 0;
};
constexpr int RING = 16;
constexpr size_t PEER_HEADER = 4096;         // flags[2][K2_MAX_PEERS] + error word, then the float buffers

struct IngestScratch {
    DevBuf<char> text;
    DevBuf<unsigned char> nl, state, tmp;
    DevBuf<int32_t> keep, pos;
    DevBuf<int64_t> nlpos;
    DevBuf<unsigned long long> scal;
    DevBuf<double> cols[8];
    void release() {
        text.release(); nl.release(); state.release(); tmp.release(); keep.release(); pos.release(); nlpos.release();
        scal.release();
        for (auto &c : cols) c.release();
    }
};

struct prb_engine {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaDeviceProp prop{};

    // line list
    int64_t n_lines = 0, n_alloc = 0;
    int n_groups = 0;
    DevBuf<double> nu0, s296, gair, gself, elower, nair, delta, einstein_a;
    DevBuf<int32_t> group;
    bool has_group = false;
    double s_max = 0;
    bool lines_set = false;
    // grouped line list (prb_upload_line_groups): group g = device entries [seg[g], seg[g] + seg_cnt[g]), ascending within
    // the group, segments 4-aligned; empty when the list is one globally ascending run (prb_upload_lines)
    std::vector<int64_t> seg, seg_cnt;
    bool group_rows_valid = false;   // out64 holds the per-group rows of the last prb_line_sum_groups

    // grid
    double range_min = 0, res = 0;
    int64_t n_total = 0, i_begin = 0, i_end = 0;
    bool grid_set = false;
    DevBuf<int32_t> idx;

    // per-layer
    DevBuf<float4> recA, recB;
    DevBuf<float> recD;
    int64_t rec_slots = 0;        // the record arrays hold rec_slots layers of n_alloc records each
    DevBuf<GroupParams> gp;       // n_layers * n_groups
    DevBuf<DevState> st;          // one per layer
    K1Table k1_host;              // K1's layer table (passed by value as a kernel parameter)
    DevBuf<K2Layer> k2tab;
    LayerJob last;
    int k2_variant = PRB_K2_CLASSED, k2_ppt = 0;
    // PRB_K2_FARFIELD: per span length (index 0: 128 points, P = 4; index 1: 256 points, P = 8) the Lagrange weights
    // [span][K2_FAR_NODES] and the FP32 node offsets (built at prb_create)
    DevBuf<double> far_lag[2];
    float far_delta[2][K2_FAR_NODES] = {};
    DevBuf<double> far_lag2[2];                       // level 2: domains of K2_FAR2_SPANS spans
    float far_delta2[2][K2_FAR_NODES] = {};
    int64_t narrow_wm = 100;     // windows with W-2 below this use k2_narrow
    bool batch_layers = true;    // prb_atmosphere: one K1 launch + one K2 launch per kernel class
    bool k3_tma = true;          // layer fold: k matrix staged by TMA (k3_fold_tma) instead of register-held loads
    bool point_kernel = true;    // windows up to 511 points: k2_point instead of k2_narrow
    bool fuse_single = true;     // single wide layer: layer physics + peer stores in K2's epilogue
    bool split_tiles = false;    // PRB_OPT_SPLIT_TILES: short K2 launches split every tile into line-range parts
    DevBuf<double> part_sums;    // [items][parts][tile] FP64 partials of such a launch
    DevBuf<unsigned int> part_count;
    int64_t rec_budget_mb = 0;   // 0 = auto (a quarter of the free memory)
    PeerState peer;
    DevBuf<unsigned int> peer_err;
    IngestScratch ingest;
    DevBuf<int2> tile_bounds_buf[2];
    int tile_bounds_next = 0;
    int extra_launches = 0;                           // helper kernels launched inside run_line_sum (counted per call)
    // pipelined host upload (prb_gas_cell_host)
    cudaStream_t copy_stream = nullptr, stream2 = nullptr;
    std::vector<cudaEvent_t> pipe_ev;
    unsigned long long *pin_scal = nullptr;           // pinned: [0] max|S296| bits, [1] validation flags
    DevBuf<unsigned long long> dev_scal;
    // pinned ring of single-layer K2 table rows (prb_line_sum_dev is enqueue-only)
    unsigned char *blk_h = nullptr;                   // pinned staging of prb_atmosphere's small tables
    size_t blk_cap = 0;
    DevBuf<unsigned char> blk_d;
    K2Layer *ring_h = nullptr;
    DevBuf<K2Layer> ring_d;
    cudaEvent_t ring_ev[RING] = {};
    int ring_next = 0;

    // resident xsc tables and their per-layer mole fractions for the next prb_atmosphere / prb_gas_cell_host
    XscTable xsc[K2_MAX_XSC];
    int n_xsc = 0;
    DevBuf<double> xsc_rows;                          // [n_xsc][xsc_ld] on the owned chunk
    int64_t xsc_ld = 0;
    bool xsc_rows_valid = false;
    int64_t xsc_sig[3] = {-1, -1, -1};                // (i_begin, i_end, n_total) the rows were built for
    int xsc_build_launches = 0;                       // resampling kernels enqueued so far (a running count)
    std::vector<double> xsc_conc;                     // [xsc_conc_layers][n_xsc]
    int xsc_conc_layers = 0;
    std::vector<double> line_lo, line_hi;             // per-layer line ranges of the next prb_atmosphere calls (may be empty)
    // the water-vapour continuum of the next prb_atmosphere / prb_gas_cell_host calls (prb_set_continuum); empty: none
    std::vector<double> cont_tab;                     // table_nu | c_self | c_foreign | t_exp
    double cont_t_ref = 0, cont_p_ref = 0;
    std::vector<double> cont_x;                       // mole fraction per layer
    DevBuf<double> cont_tab_dev;
    DevBuf<float> cont_rows;                          // [3][kmat_ld]: C_s, C_f, n on the owned chunk
    std::vector<double> cont_rows_tab;                // the table the rows hold (kept when the continuum is cleared)
    double cont_sig[5] = {};                          // (i_begin, i_end, n_total, range_min, range_max) of the rows
    DevBuf<ContLayer> cont_layers;

    // outputs / scratch
    DevBuf<double> out64;
    DevBuf<double> scratch_a, scratch_b, scratch_c, scratch_d, scratch_w;
    // atmosphere
    DevBuf<float> kmat, rad, trans;
    float *res_rad = nullptr, *res_trans = nullptr;   // where the last prb_atmosphere left its spectra
    float *read_stage = nullptr;                      // pinned staging of prb_atmosphere_read
    size_t read_stage_cap = 0;
    float *host_rad_dev = nullptr, *host_trans_dev = nullptr;   // device views of the caller's pinned result buffers
    int64_t host_result_len = 0;
    int last_launches = 0;                            // kernels launched by the last prb_atmosphere
    DevBuf<FoldLayer> fold;
    int64_t kmat_ld = 0;
    int atm_layers = 0;
    // the last column's layer constants and fold policy, for prb_atmosphere_fluxes
    std::vector<double> atm_depth, atm_t;
    double atm_t_surface = 0, atm_range_max = 0;
    float atm_nu_interp_min = 1e30f;                  // Planck interpolated above this (k3_fold_tma), else per point
    DevBuf<FluxLayer> flux_layers;
    DevBuf<double> flux_part, flux_out;
    DevBuf<float> flux_rows;
    DevBuf<double> band_part, band_out;               // prb_atmosphere_band_fluxes: per-segment level sums, band totals
    DevBuf<int32_t> band_tab;                         // its span, segment, band and strip tables
    // the flux calls' boundaries (prb_set_flux_boundaries); an empty table and t_top = 0: a black surface, 0 at the top
    std::vector<double> bnd_tab;                      // table_nu | table_emissivity
    int bnd_reflection = PRB_REFLECT_LAMBERTIAN;
    double bnd_t_top = 0;
    DevBuf<double> bnd_tab_dev;
    DevBuf<float> flux_eps;                           // the emissivity on the owned chunk
    // the flux calls' solar beam (prb_set_solar_source); an empty table: no Sun
    std::vector<double> sun_tab;                      // table_nu | table_irradiance
    double sun_mu = 1;
    DevBuf<double> sun_tab_dev;
    DevBuf<float> sun_nd;                             // -depth_l log2(e) / mu_sun per layer
    // optional stage timing of prb_atmosphere (CUDA events on the engine stream)
    bool timing = false;
    std::vector<cudaEvent_t> ev;
    float t_k1 = 0, t_k2 = 0, t_k3 = 0;
    std::vector<float> t_layer_k1, t_layer_k2;
};

static int64_t chunk_len(const prb_engine *e) { return e->i_end - e->i_begin; }

extern "C" int prb_abi_version(void) { return PRB_ABI_VERSION; }
extern "C" const char *prb_last_error(void) { return g_err.c_str(); }

static int build_far_table(prb_engine *e);

extern "C" int prb_create(int device, prb_engine **out) {
    if (!out) return fail(PRB_ERR_ARG, "prb_create: out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || count == 0)
        return fail(PRB_ERR_NODEVICE, std::string("prb_create: no CUDA device (") + cudaGetErrorString(ce) +
                                          "); libpyrad_b200 has no CPU fallback");
    if (device < 0 || device >= count) return fail(PRB_ERR_ARG, "prb_create: device ordinal out of range");
    CK(cudaSetDevice(device));
    prb_engine *e = new prb_engine();
    e->device = device;
    k1_fill_constants(e->k1_host);
    if (cudaGetDeviceProperties(&e->prop, device) != cudaSuccess) {
        delete e;
        return fail(PRB_ERR_CUDA, "prb_create: cudaGetDeviceProperties failed");
    }
    if (e->prop.major != 10) {
        char b[256];
        snprintf(b, sizeof b, "prb_create: device is sm_%d%d; this library only carries sm_100a code (no fallback)",
                 e->prop.major, e->prop.minor);
        delete e;
        return fail(PRB_ERR_NODEVICE, b);
    }
    if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete e;
        return fail(PRB_ERR_CUDA, "prb_create: cudaStreamCreate failed");
    }
    // opt-in shared memory of the kernels that stage through it (per device, so here and not in process-wide statics)
    cudaError_t ae = cudaSuccess;
    auto want = [&](const void *fn, size_t bytes) {
        if (ae == cudaSuccess) ae = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    };
    want((const void *)k2_line_sum<2>, K2_SMEM_BYTES<2>(true));
    want((const void *)k2_line_sum<4>, K2_SMEM_BYTES<4>(true));
    want((const void *)k2_line_sum<8>, K2_SMEM_BYTES<8>(true));
    want((const void *)k2_line_sum<16>, K2_SMEM_BYTES<16>(true));
    want((const void *)k2_line_sum_far<4>, K2_SMEM_BYTES<4>(true));
    want((const void *)k2_line_sum_far<8>, K2_SMEM_BYTES<8>(true));
    want((const void *)k2_line_sum<2, true>, K2_SMEM_BYTES<2>(true));
    want((const void *)k2_line_sum<4, true>, K2_SMEM_BYTES<4>(true));
    want((const void *)k2_line_sum<8, true>, K2_SMEM_BYTES<8>(true));
    want((const void *)k2_line_sum<16, true>, K2_SMEM_BYTES<16>(true));
    want((const void *)k2_line_sum_far<4, true>, K2_SMEM_BYTES<4>(true));
    want((const void *)k2_line_sum_far<8, true>, K2_SMEM_BYTES<8>(true));
    want((const void *)k2_point, sizeof(KPSmem));
    want((const void *)k3_fold_tma, sizeof(K3TSmem));
    if (ae != cudaSuccess) {
        cudaStreamDestroy(e->stream);
        delete e;
        return fail(PRB_ERR_CUDA, std::string("prb_create: cudaFuncSetAttribute failed: ") + cudaGetErrorString(ae));
    }
    if (cudaSetDevice(device) != cudaSuccess || build_far_table(e) != PRB_OK) {
        e->far_lag[0].release(); e->far_lag[1].release(); e->far_lag2[0].release(); e->far_lag2[1].release();
        cudaStreamDestroy(e->stream);
        delete e;
        return fail(PRB_ERR_CUDA, "prb_create: far-field table upload failed");
    }
    *out = e;
    return PRB_OK;
}

static void peer_release(prb_engine *e) {
    PeerState &ps = e->peer;
    for (int r = 0; r < ps.world; ++r)
        if (ps.connected && r != ps.rank && ps.base[r]) cudaIpcCloseMemHandle(ps.base[r]);
    if (ps.local) cudaFree(ps.local);
    ps = PeerState{};
}

extern "C" int prb_destroy(prb_engine *e) {
    if (!e) return PRB_OK;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    e->nu0.release(); e->s296.release(); e->gair.release(); e->gself.release();
    e->elower.release(); e->nair.release(); e->delta.release(); e->group.release(); e->einstein_a.release();
    e->idx.release(); e->recA.release(); e->recB.release(); e->recD.release(); e->gp.release(); e->st.release();
    e->out64.release(); e->scratch_a.release(); e->scratch_b.release(); e->scratch_c.release();
    e->scratch_d.release(); e->scratch_w.release();
    e->kmat.release(); e->rad.release(); e->trans.release(); e->fold.release();
    e->flux_layers.release(); e->flux_part.release(); e->flux_out.release(); e->flux_rows.release();
    e->band_part.release(); e->band_out.release(); e->band_tab.release();
    e->bnd_tab_dev.release(); e->flux_eps.release();
    e->sun_tab_dev.release(); e->sun_nd.release();
    e->k2tab.release(); e->ring_d.release(); e->peer_err.release();
    if (e->blk_h) cudaFreeHost(e->blk_h);
    if (e->read_stage) cudaFreeHost(e->read_stage);
    e->blk_d.release();
    e->ingest.release();
    e->tile_bounds_buf[0].release(); e->tile_bounds_buf[1].release();
    e->far_lag[0].release(); e->far_lag[1].release(); e->far_lag2[0].release(); e->far_lag2[1].release();
    e->dev_scal.release();
    e->part_sums.release(); e->part_count.release();
    e->xsc_rows.release();
    for (auto &x : e->xsc) { x.fx.release(); x.fy.release(); }
    if (e->pin_scal) cudaFreeHost(e->pin_scal);
    for (auto x : e->pipe_ev) cudaEventDestroy(x);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->stream2) cudaStreamDestroy(e->stream2);
    if (e->ring_h) { cudaFreeHost(e->ring_h); for (auto x : e->ring_ev) if (x) cudaEventDestroy(x); }
    peer_release(e);
    for (auto x : e->ev) cudaEventDestroy(x);
    cudaStreamDestroy(e->stream);
    delete e;
    return PRB_OK;
}

extern "C" void *prb_stream(prb_engine *e) { return e ? (void *)e->stream : nullptr; }

// Page-locked host memory for callers that keep line columns / result buffers around (the host mirror's Isotope): copies
// from and to it run at PCIe speed instead of through the driver's staging buffer.  NULL when no device is usable.
extern "C" void *prb_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
extern "C" int prb_host_free(void *p) {
    if (p && cudaFreeHost(p) != cudaSuccess) return fail(PRB_ERR_CUDA, "prb_host_free: cudaFreeHost failed");
    return PRB_OK;
}

static int report_flags(const DevState *h, int n_states) {
    unsigned int f = 0;
    for (int k = 0; k < n_states; ++k) f |= h[k].flags;
    if (f & FLAG_NONFINITE)
        return fail(PRB_ERR_RANGE, "line prepass produced a non-finite coefficient (bad line data or T/P/Q inputs)");
    if (f & FLAG_OVERFLOW)
        return fail(PRB_ERR_RANGE, "line coefficient exceeds the scaled FP32 range (window too wide or S(T)/S296 too large)");
    return PRB_OK;
}

static int check_flags(prb_engine *e, int n_states) {
    std::vector<DevState> h(n_states);
    CK(cudaMemcpyAsync(h.data(), e->st.p, sizeof(DevState) * n_states, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return report_flags(h.data(), n_states);
}

extern "C" int prb_synchronize(prb_engine *e) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
    return PRB_OK;
}

// Roofline denominators measured here and now (k9_peaks.cuh): FP32 lane-FMAs per second of the packed FFMA2 and the
// scalar FFMA instruction streams (best of `reps` launches each, CUDA events on the engine stream) and the float4 copy
// bandwidth (read + write bytes) over a buffer well beyond the L2.
extern "C" int prb_measure_peaks(prb_engine *e, double *ffma2_lane_fma_per_s, double *ffma_lane_fma_per_s,
                                 double *copy_bytes_per_s) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    CK(cudaSetDevice(e->device));
    const int sms = e->prop.multiProcessorCount;
    const int grid = sms * 8, iters = 4096, reps = 5;
    DevBuf<float> sink;
    CK(sink.ensure((size_t)grid * 256));
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    auto best_ms = [&](const std::function<void()> &launch, float *out) -> int {
        float best = 1e30f;
        for (int r = 0; r < reps + 1; ++r) {                       // the first launch warms clocks and instruction cache
            CK(cudaEventRecord(a, e->stream));
            launch();
            CK(cudaGetLastError());
            CK(cudaEventRecord(b, e->stream));
            CK(cudaEventSynchronize(b));
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, a, b));
            if (r) best = std::min(best, ms);
        }
        *out = best;
        return PRB_OK;
    };
    int rc;
    float ms = 0;
    const double lane_fma = (double)grid * 256 * (double)iters * K9_UNROLL * K9_CHAINS * 2;
    if (ffma2_lane_fma_per_s) {
        if ((rc = best_ms([&] { k9_ffma2_peak<<<grid, 256, 0, e->stream>>>(sink.p, iters, 1.5f); }, &ms))) return rc;
        *ffma2_lane_fma_per_s = lane_fma / (ms * 1e-3);
    }
    if (ffma_lane_fma_per_s) {
        if ((rc = best_ms([&] { k9_ffma_peak<<<grid, 256, 0, e->stream>>>(sink.p, iters, 1.5f); }, &ms))) return rc;
        *ffma_lane_fma_per_s = lane_fma / (ms * 1e-3);
    }
    if (copy_bytes_per_s) {
        const int64_t n4 = (int64_t)64 << 20;                      // 1 GiB each way
        DevBuf<float4> src, dst;
        CK(src.ensure((size_t)n4));
        CK(dst.ensure((size_t)n4));
        CK(cudaMemsetAsync(src.p, 0, sizeof(float4) * n4, e->stream));
        if ((rc = best_ms([&] { k9_copy<<<sms * 16, 256, 0, e->stream>>>(src.p, dst.p, n4); }, &ms))) return rc;
        *copy_bytes_per_s = 2.0 * sizeof(float4) * (double)n4 / (ms * 1e-3);
        src.release();
        dst.release();
    }
    sink.release();
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    return PRB_OK;
}

extern "C" int prb_device_info(prb_engine *e, int *sm_count, int *cc_major, int *cc_minor, int *sm_clock_khz,
                               size_t *free_bytes, size_t *total_bytes) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    CK(cudaSetDevice(e->device));
    if (sm_count) *sm_count = e->prop.multiProcessorCount;
    if (cc_major) *cc_major = e->prop.major;
    if (cc_minor) *cc_minor = e->prop.minor;
    if (sm_clock_khz) {
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, e->device);
        *sm_clock_khz = khz;
    }
    if (free_bytes || total_bytes) {
        size_t f = 0, t = 0;
        CK(cudaMemGetInfo(&f, &t));
        if (free_bytes) *free_bytes = f;
        if (total_bytes) *total_bytes = t;
    }
    return PRB_OK;
}

// classed kernels (per-warp window classes, thread-per-point kernels for narrow windows): every variant but GENERAL
static inline bool k2_classed(const prb_engine *e) { return e->k2_variant != PRB_K2_GENERAL; }

// Chebyshev nodes of a span on [-0.5, span - 0.5] as FP32 offsets from its first point, and the Lagrange weight of
// every node at every point (FP64, built from the ROUNDED offsets so that kernel and table agree exactly).
static int build_far_table(prb_engine *e) {
    const double pi = 3.14159265358979323846;
    auto build = [&](int span, float *delta, DevBuf<double> &dev) -> int {
        double node[K2_FAR_NODES];
        for (int k = 0; k < K2_FAR_NODES; ++k) {
            delta[k] = (float)(0.5 * (span - 1) + 0.5 * span * std::cos((2 * k + 1) * pi / (2 * K2_FAR_NODES)));
            node[k] = (double)delta[k];
        }
        std::vector<double> lag((size_t)span * K2_FAR_NODES);      // node-major: [node][point]
        for (int i = 0; i < span; ++i)
            for (int k = 0; k < K2_FAR_NODES; ++k) {
                double w = 1.0;
                for (int j = 0; j < K2_FAR_NODES; ++j)
                    if (j != k) w *= ((double)i - node[j]) / (node[k] - node[j]);
                lag[(size_t)k * span + i] = w;
            }
        CK(dev.ensure(lag.size()));
        CK(cudaMemcpy(dev.p, lag.data(), sizeof(double) * lag.size(), cudaMemcpyHostToDevice));
        return PRB_OK;
    };
    for (int t = 0; t < 2; ++t) {
        const int span = t == 0 ? 128 : 256;
        int rc = build(span, e->far_delta[t], e->far_lag[t]);
        if (rc == PRB_OK) rc = build(span * K2_FAR2_SPANS, e->far_delta2[t], e->far_lag2[t]);
        if (rc) return rc;
    }
    return PRB_OK;
}

// PRB_K2_FARFIELD launches k2_line_sum<P, true> where a table exists (P = 4, 8); other P run the exact kernel.
template <int P>
static bool far_args(const prb_engine *e, K2Args &a) {
    if (a.variant != PRB_K2_FARFIELD || (P != 4 && P != 8)) return false;
    const int t = P == 4 ? 0 : 1;
    a.far_lag = e->far_lag[t].p;
    a.far_lag2 = e->far_lag2[t].p;
    for (int k = 0; k < K2_FAR_NODES; ++k) { a.far_delta[k] = e->far_delta[t][k]; a.far_delta2[k] = e->far_delta2[t][k]; }
    return true;
}

extern "C" int prb_set_k2_variant(prb_engine *e, int variant, int ppt) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (variant != PRB_K2_GENERAL && variant != PRB_K2_CLASSED && variant != PRB_K2_FARFIELD)
        return fail(PRB_ERR_ARG, "unknown K2 variant");
    if (ppt != 0 && ppt != 2 && ppt != 4 && ppt != 8 && ppt != 16)
        return fail(PRB_ERR_ARG, "points_per_thread must be 0 (auto), 2, 4, 8 or 16");
    e->k2_variant = variant;
    e->k2_ppt = ppt;
    return PRB_OK;
}

// ------------------------------------------------------------------------------------ lines
// Device storage for n lines: SoA columns, grid indices and one layer of K2 records, all with padding records
// (TMA copies are 16-byte granular) and a length that is a multiple of 4 so every per-layer slice of the record
// arrays starts 16-byte aligned.
static int alloc_line_storage(prb_engine *e, int64_t n) {
    const int64_t na = (n + 16 + 3) & ~int64_t(3);
    DevBuf<double> *cols[8] = {&e->nu0, &e->s296, &e->gair, &e->gself, &e->elower, &e->nair, &e->delta, &e->einstein_a};
    for (int c = 0; c < 8; ++c) CK(cols[c]->ensure(na));
    CK(e->idx.ensure(na));
    CK(e->recA.ensure(na));
    CK(e->recB.ensure(na));
    CK(e->recD.ensure(na));
    e->rec_slots = (int64_t)(std::min(e->recA.n, std::min(e->recB.n, e->recD.n)) / (size_t)na);
    e->n_alloc = na;
    return PRB_OK;
}

extern "C" int prb_upload_lines(prb_engine *e, int64_t n, const double *nu0, const double *s296,
                                const double *gamma_air, const double *gamma_self, const double *elower,
                                const double *n_air, const double *delta_air, const int32_t *group,
                                int32_t n_groups) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n < 0 || n > 2000000000LL) return fail(PRB_ERR_ARG, "prb_upload_lines: n out of range");
    if (n_groups < 1) return fail(PRB_ERR_ARG, "prb_upload_lines: n_groups must be >= 1");
    if (n > 0 && (!nu0 || !s296 || !gamma_air || !gamma_self || !elower || !n_air || !delta_air))
        return fail(PRB_ERR_ARG, "prb_upload_lines: NULL column");
    CK(cudaSetDevice(e->device));
    int rc = alloc_line_storage(e, n);
    if (rc) return rc;
    const int64_t na = e->n_alloc;
    DevBuf<double> *cols[7] = {&e->nu0, &e->s296, &e->gair, &e->gself, &e->elower, &e->nair, &e->delta};
    const double *src[7] = {nu0, s296, gamma_air, gamma_self, elower, n_air, delta_air};
    if (!e->pin_scal) CK(cudaMallocHost((void **)&e->pin_scal, 64));
    CK(e->dev_scal.ensure(8));
    e->has_group = group != nullptr;
    if (group) CK(e->group.ensure(na));
    if (n) {
        CK(cudaMemsetAsync(e->dev_scal.p, 0, 2 * sizeof(unsigned long long), e->stream));
        CK(cudaMemcpyAsync(cols[0]->p, src[0], sizeof(double) * n, cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemcpyAsync(cols[1]->p, src[1], sizeof(double) * n, cudaMemcpyHostToDevice, e->stream));
        if (group) CK(cudaMemcpyAsync(e->group.p, group, sizeof(int32_t) * n, cudaMemcpyHostToDevice, e->stream));
        // the checks of the line list -- ascending nu0, group ids in range -- and max|S296| run on the device over the
        // columns just uploaded, while the other five cross the bus (a host pass over the caller's arrays costs as much
        // as their PCIe time)
        k0_validate_lines<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(e->nu0.p, group ? e->group.p : nullptr, n, n_groups,
                                                                            reinterpret_cast<unsigned int *>(e->dev_scal.p + 1));
        k0_absmax<<<e->prop.multiProcessorCount * 4, 256, 0, e->stream>>>(e->s296.p, n, e->dev_scal.p);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(e->pin_scal, e->dev_scal.p, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream));
        for (int c = 2; c < 7; ++c)
            CK(cudaMemcpyAsync(cols[c]->p, src[c], sizeof(double) * n, cudaMemcpyHostToDevice, e->stream));
    }
    CK(cudaStreamSynchronize(e->stream));
    e->lines_set = false;
    double smax = 0;
    if (n) {
        memcpy(&smax, e->pin_scal, sizeof(double));
        const unsigned int vf = (unsigned int)e->pin_scal[1];
        if (vf & 1u) return fail(PRB_ERR_ARG, "prb_upload_lines: nu0 must be ascending");
        if (vf & 2u) return fail(PRB_ERR_ARG, "prb_upload_lines: group id out of range");
    }
    e->n_lines = n;
    e->n_groups = n_groups;
    e->s_max = smax;
    e->lines_set = true;
    e->grid_set = false;
    e->last.valid = false;
    e->seg.clear();
    e->seg_cnt.clear();
    e->group_rows_valid = false;
    return PRB_OK;
}

// Grouped line list (SURVEY 8(b): per-group output rows in one pass).  The host object model holds one line list per
// isotopologue, each ascending in nu0 (pyradClasses.py:350-359); they are uploaded as they are -- concatenated, no merge
// sort -- and every group becomes its own work-item row of ONE K2 launch (prb_line_sum_groups), walking only its own
// lines.  Segments start 16-byte aligned on the device (the TMA staging of K2 aligns its first record down by up to
// three entries); the gap entries carry group -1 and are inert.
extern "C" int prb_upload_line_groups(prb_engine *e, int32_t n_groups, const int64_t *counts,
                                      const double *const *nu0, const double *const *s296,
                                      const double *const *gamma_air, const double *const *gamma_self,
                                      const double *const *elower, const double *const *n_air,
                                      const double *const *delta_air) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n_groups < 1 || !counts) return fail(PRB_ERR_ARG, "prb_upload_line_groups: bad group count");
    if (!nu0 || !s296 || !gamma_air || !gamma_self || !elower || !n_air || !delta_air)
        return fail(PRB_ERR_ARG, "prb_upload_line_groups: NULL column table");
    int64_t n = 0;
    for (int g = 0; g < n_groups; ++g) {
        if (counts[g] < 0) return fail(PRB_ERR_ARG, "prb_upload_line_groups: negative line count");
        if (counts[g] > 0 && (!nu0[g] || !s296[g] || !gamma_air[g] || !gamma_self[g] || !elower[g] || !n_air[g] || !delta_air[g]))
            return fail(PRB_ERR_ARG, "prb_upload_line_groups: NULL column");
        n += counts[g];
    }
    if (n > 2000000000LL) return fail(PRB_ERR_ARG, "prb_upload_line_groups: too many lines");
    CK(cudaSetDevice(e->device));
    std::vector<int64_t> seg(n_groups + 1, 0), cnt(n_groups, 0);
    for (int g = 0; g < n_groups; ++g) {
        cnt[g] = counts[g];
        seg[g + 1] = (seg[g] + cnt[g] + 3) & ~int64_t(3);
    }
    const int64_t n_dev = seg[n_groups];
    int rc = alloc_line_storage(e, n_dev);
    if (rc) return rc;
    const int64_t na = e->n_alloc;
    CK(e->group.ensure(na));
    DevBuf<double> *cols[7] = {&e->nu0, &e->s296, &e->gair, &e->gself, &e->elower, &e->nair, &e->delta};
    const double *const *src[7] = {nu0, s296, gamma_air, gamma_self, elower, n_air, delta_air};
    if (!e->pin_scal) CK(cudaMallocHost((void **)&e->pin_scal, 64));
    CK(e->dev_scal.ensure(8));
    CK(cudaMemsetAsync(e->dev_scal.p, 0, 2 * sizeof(unsigned long long), e->stream));
    // the S296 and nu0 columns first: their checks run on the device while the other columns cross the bus
    for (int c = 0; c < 7; ++c) {
        for (int g = 0; g < n_groups; ++g)
            if (cnt[g])
                CK(cudaMemcpyAsync(cols[c]->p + seg[g], src[c][g], sizeof(double) * cnt[g], cudaMemcpyHostToDevice, e->stream));
        if (c != 1 || !n_dev) continue;
        // group ids, gap entries, and what prb_upload_lines checks in its host pass -- max|S296| and "ascending within
        // every group" -- as device kernels over the uploaded columns (a host pass over 0.5 M lines costs as much as
        // their PCIe time): no host vector of group ids, no second read of the caller's columns
        CK(cudaMemsetAsync(e->group.p, 0xFF, sizeof(int32_t) * n_dev, e->stream));
        for (int g = 0; g < n_groups; ++g) {
            if (!cnt[g]) continue;
            const unsigned nb = (unsigned)((cnt[g] + 255) / 256);
            k0_set_group<<<nb, 256, 0, e->stream>>>(e->group.p + seg[g], cnt[g], g);
            k0_validate_lines<<<nb, 256, 0, e->stream>>>(e->nu0.p + seg[g], nullptr, cnt[g], n_groups,
                                                        reinterpret_cast<unsigned int *>(e->dev_scal.p + 1));
        }
        k0_fill_gaps<<<(unsigned)((n_dev + 255) / 256), 256, 0, e->stream>>>(e->nu0.p, e->s296.p, e->group.p, n_dev);
        k0_absmax<<<e->prop.multiProcessorCount * 4, 256, 0, e->stream>>>(e->s296.p, n_dev, e->dev_scal.p);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(e->pin_scal, e->dev_scal.p, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream));
    }
    CK(cudaStreamSynchronize(e->stream));
    e->lines_set = false;
    double smax = 0;
    if (n_dev) {
        memcpy(&smax, e->pin_scal, sizeof(double));
        if ((unsigned int)e->pin_scal[1] & 1u)
            return fail(PRB_ERR_ARG, "prb_upload_line_groups: nu0 must be ascending within every group");
    }
    e->has_group = true;
    e->n_lines = n_dev;
    e->n_groups = n_groups;
    e->s_max = smax;
    e->lines_set = true;
    e->grid_set = false;
    e->last.valid = false;
    e->seg.assign(seg.begin(), seg.end() - 1);
    e->seg_cnt = cnt;
    e->group_rows_valid = false;
    return PRB_OK;
}

// ------------------------------------------------------------------------------------ grid
extern "C" int prb_set_grid(prb_engine *e, double range_min, double res, int64_t n_total, int64_t i_begin,
                            int64_t i_end) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (!e->lines_set) return fail(PRB_ERR_STATE, "prb_set_grid: upload lines first");
    if (!(res > 0) || n_total < 0 || i_begin < 0 || i_end < i_begin || i_end > n_total)
        return fail(PRB_ERR_ARG, "prb_set_grid: bad grid");
    if (n_total > 2000000000LL) return fail(PRB_ERR_ARG, "prb_set_grid: n_total too large");
    CK(cudaSetDevice(e->device));
    const int64_t na = e->n_alloc;
    k0_line_index<<<(unsigned)((na + 255) / 256), 256, 0, e->stream>>>(e->nu0.p, e->n_lines, 0, na, range_min, res,
                                                                      e->idx.p);
    CK(cudaGetLastError());                                     // enqueue only: the indices never visit the host
    e->range_min = range_min;
    e->res = res;
    e->n_total = n_total;
    e->i_begin = i_begin;
    e->i_end = i_end;
    e->grid_set = true;
    e->last.valid = false;
    e->xsc_rows_valid = false;
    e->group_rows_valid = false;
    return PRB_OK;
}

// ------------------------------------------------------------------------------------ K1
static int build_group_params(int n_groups, double T, const double *conc, const double *molmass, const double *q_t,
                              const double *q_296, const double *weight, GroupParams *out, double *w_max) {
    double wm = 0;
    for (int g = 0; g < n_groups; ++g) {
        const double m = molmass[g] / 1000 / kAvogadro;                        // pyradClasses.py:294-296
        out[g].conc = conc[g];
        out[g].dopp = std::sqrt(2 * kBoltz * T / m / (cLight * cLight));       // pyradClasses.py:263
        out[g].qratio = q_296[g] / q_t[g];                                     // pyradIntensity.py:31
        out[g].weight = weight ? weight[g] : 1.0;
        wm = std::max(wm, std::fabs(out[g].weight));
    }
    *w_max = wm;
    return PRB_OK;
}

static double pick_scale(double s_max, double w_max) {
    // Power of two that puts the strongest possible S296*weight near 2^10: typical A = S*eta*h/pi/res^2
    // then sits around 2^25..2^35, leaving headroom for A*q^2 (q = d^2+B up to ~2^30) and ~2^-126 as the floor.
    const double m = s_max * w_max;
    if (!(m > 0) || !std::isfinite(m)) return 1.0;
    return std::ldexp(1.0, 10 - std::ilogb(m));
}

static LayerConsts layer_consts(double T, double P, double res) {
    LayerConsts lc;
    lc.log_t0_over_t = std::log(kT0 / T);
    lc.inv_t_minus_inv_t0 = 1.0 / T - 1.0 / kT0;
    lc.inv_res2 = 1.0 / (res * res);
    lc.res2 = res * res;
    lc.p_over_p0 = P / kP0;
    const double c2 = cLight * hPlanck * 100 / kBoltz;
    lc.neg_c2_over_t = -c2 / T;
    lc.neg_c2_over_t0 = -c2 / kT0;
    return lc;
}

static int check_segment(prb_engine *e, int64_t wm) {
    // FP32 offsets must be exact integers: chunk + tile rounding + both windows below 2^24.
    if (chunk_len(e) + 2 * wm + 8192 >= (int64_t(1) << 24))
        return fail(PRB_ERR_RANGE, "owned grid chunk plus cutoff windows exceeds 2^24 points; shard the grid "
                                   "(prb_set_grid i_begin/i_end) into smaller chunks");
    return PRB_OK;
}

static int pick_ppt(const prb_engine *e, int64_t wm) {
    if (e->k2_ppt) return e->k2_ppt;
    // a warp spans 32*P points: keep the span well inside the window so most lines cover it fully
    // (thresholds measured per layer on B200, profiles/r01_k2_experiments.txt)
#ifndef PRB_FAR_P8_MIN
#define PRB_FAR_P8_MIN 3072
#endif
    // (far-field variant: a 128-point span halves the near zone and the partly covered lines at twice the node
    // evaluations, which pays up to wider windows than in the exact kernel: cfg4 K2 67.3 ms with the 256-point span
    // from W-2 >= 1024, 66.2 / 65.5 / 64.9 / 65.2 / 64.7 from 1536 / 2048 / 3072 / 4096 / never)
    if (e->k2_variant == PRB_K2_FARFIELD) return wm >= PRB_FAR_P8_MIN ? 8 : (wm >= 256 ? 4 : 2);
    if (wm >= 1024) return 8;
    if (wm >= 256) return 4;
    return 2;
}

// Window, kernel class and K2 line range of one layer on the owned chunk.
static LayerJob plan_job(const prb_engine *e, double T, double P, int64_t W, double scale) {
    LayerJob j;
    j.T = T; j.P = P; j.W = W; j.scale = scale;
    j.wm = std::max<int64_t>(W - 2, 0);
    // The prepass covers the whole uploaded list and K2's producer searches all of it for every tile: callers upload
    // the lines that can reach the owned chunk (ShardPlan.subset), so narrowing the range here bought nothing and cost
    // a device-to-host copy of the index array plus a synchronisation in every prb_set_grid.
    j.l0 = 0;
    j.l1 = e->n_lines;
    // kernel kind: 0 = k2_line_sum (wide), 2 = k2_point (table-driven thread-per-point, 16 <= W-2 <= 511),
    // 1 = k2_narrow (binary-search thread-per-point: windows of a few points, where building the table costs more
    //     than it saves -- measured on B200 -- and forced thresholds above 511)
    j.narrow = 0;
    if (k2_classed(e) && j.wm < e->narrow_wm)
        j.narrow = (e->point_kernel && j.wm >= KP_MIN_WM && j.wm <= KP_MAX_WM) ? 2 : 1;
    j.ppt = pick_ppt(e, j.wm);
    j.valid = true;
    return j;
}

static int ensure_records(prb_engine *e, int64_t slots) {
    if (slots <= e->rec_slots) return PRB_OK;
    const size_t na = (size_t)e->n_alloc;
    CK(e->recA.ensure(na * slots));
    CK(e->recB.ensure(na * slots));
    CK(e->recD.ensure(na * slots));
    e->rec_slots = slots;
    return PRB_OK;
}

static void fill_k1_row(const prb_engine *e, const LayerJob &j, K1Layer &t) {
    const size_t na = (size_t)e->n_alloc;
    t.T = j.T; t.P = j.P;
    t.lc = layer_consts(j.T, j.P, e->res);
    t.scale = j.scale;
    t.scale_dev = j.scale_dev;
    t.wm = (double)j.wm;
    t.gp = j.gp_dev;
    t.recA = e->recA.p + na * j.slot;
    t.recB = e->recB.p + na * j.slot;
    t.recD = e->recD.p + na * j.slot;
    t.st = j.st_dev;
    t.narrow = j.narrow;
    t.pad = 0;
}

// K1 for jobs[0..n): ONE launch per K1_MAX_LAYERS layers over the union of their line ranges, every thread walking
// the layers.  The layer table is a kernel parameter (constant bank), so nothing has to be uploaded first.
static int run_prepass(prb_engine *e, const LayerJob *jobs, int n, DebugOut dbg, int *launches = nullptr) {
    for (int k0 = 0; k0 < n; k0 += K1_MAX_LAYERS) {
        const int m = std::min(n - k0, K1_MAX_LAYERS);
        K1Table &tab = e->k1_host;
        tab.n = m;
        tab.pad = 0;
        int64_t l0 = jobs[k0].l0, l1 = jobs[k0].l1;
        for (int k = 0; k < m; ++k) {
            fill_k1_row(e, jobs[k0 + k], tab.rows[k]);
            l0 = std::min(l0, jobs[k0 + k].l0);
            l1 = std::max(l1, jobs[k0 + k].l1);
        }
        const int64_t kb = l0 & ~int64_t(3);
        const int64_t ke = std::min<int64_t>(l1 + 8, e->n_alloc);
        const int64_t cnt = ke - kb;
        if (cnt > 0) {
            LinesSoA L{e->nu0.p, e->s296.p, e->gair.p, e->gself.p, e->elower.p, e->nair.p, e->delta.p,
                       e->has_group ? e->group.p : nullptr};
            k1_prepass<false><<<(unsigned)((cnt + 255) / 256), 256, 0, e->stream>>>(L, e->idx.p, tab, kb, ke, e->n_lines,
                                                                            e->i_begin, dbg);
            CK(cudaGetLastError());
            if (launches) ++*launches;
            // layers that use only the lines of their own range (prb_set_layer_line_range): blank the records of the others
            LineRangeTable lr;
            lr.n = 0; lr.pad = 0;
            const size_t na = (size_t)e->n_alloc;
            for (int k = 0; k < m; ++k) {
                const LayerJob &j = jobs[k0 + k];
                if (!j.filter) continue;
                LineRangeRow &r = lr.rows[lr.n++];
                r.recA = e->recA.p + na * j.slot;
                r.recB = e->recB.p + na * j.slot;
                r.recD = e->recD.p + na * j.slot;
                r.lo = j.nu_lo; r.hi = j.nu_hi;
                r.narrow = j.narrow; r.pad = 0;
            }
            if (lr.n) {
                k1_mask_line_range<<<lr.n, 256, 0, e->stream>>>(e->nu0.p, 0, e->n_lines, lr);
                CK(cudaGetLastError());
                if (launches) ++*launches;
            }
        }
    }
    return PRB_OK;
}

extern "C" int prb_layer_prepass(prb_engine *e, double T, double P, int32_t n_groups, const double *conc,
                                 const double *molmass, const double *q_t, const double *q_296,
                                 const double *weight, int64_t window_len) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (!e->grid_set) return fail(PRB_ERR_STATE, "prb_layer_prepass: set the grid first");
    if (n_groups != e->n_groups) return fail(PRB_ERR_ARG, "prb_layer_prepass: n_groups differs from the uploaded lines");
    if (!conc || !molmass || !q_t || !q_296) return fail(PRB_ERR_ARG, "prb_layer_prepass: NULL group array");
    if (window_len < 1) return fail(PRB_ERR_ARG, "prb_layer_prepass: window_len must be >= 1 (cutoff >= one sample)");
    if (!(T > 0) || !(P >= 0)) return fail(PRB_ERR_ARG, "prb_layer_prepass: bad T or P");
    CK(cudaSetDevice(e->device));
    int rc = check_segment(e, std::max<int64_t>(window_len - 2, 0));
    if (rc) return rc;
    std::vector<GroupParams> h(n_groups);
    double w_max = 0;
    build_group_params(n_groups, T, conc, molmass, q_t, q_296, weight, h.data(), &w_max);
    CK(e->gp.ensure(n_groups));
    CK(e->st.ensure(1));
    CK(e->k2tab.ensure(1));
    if ((rc = ensure_records(e, 1))) return rc;
    CK(cudaMemcpyAsync(e->gp.p, h.data(), sizeof(GroupParams) * n_groups, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemsetAsync(e->st.p, 0, sizeof(DevState), e->stream));
    LayerJob j = plan_job(e, T, P, window_len, pick_scale(e->s_max, w_max));
    j.gp_dev = e->gp.p;
    j.st_dev = e->st.p;
    rc = run_prepass(e, &j, 1, DebugOut{});
    if (rc) return rc;
    // (no synchronisation: a copy from pageable memory has left its source when cudaMemcpyAsync returns, and the
    // K1 layer table travels as a kernel parameter)
    e->last = j;
    e->group_rows_valid = false;
    return PRB_OK;
}

extern "C" int prb_debug_line_params(prb_engine *e, double *nu_shift, double *gamma_l, double *gamma_d, double *s_t,
                                     int32_t *regime, int64_t *index) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (!e->last.valid) return fail(PRB_ERR_STATE, "prb_debug_line_params: run prb_layer_prepass first");
    CK(cudaSetDevice(e->device));
    const int64_t n = e->n_lines, na = e->n_alloc;
    CK(e->scratch_a.ensure(na)); CK(e->scratch_b.ensure(na)); CK(e->scratch_c.ensure(na)); CK(e->scratch_d.ensure(na));
    DevBuf<int32_t> reg;
    CK(reg.ensure(na));
    CK(cudaMemsetAsync(e->scratch_a.p, 0, sizeof(double) * na, e->stream));
    CK(cudaMemsetAsync(e->scratch_b.p, 0, sizeof(double) * na, e->stream));
    CK(cudaMemsetAsync(e->scratch_c.p, 0, sizeof(double) * na, e->stream));
    CK(cudaMemsetAsync(e->scratch_d.p, 0, sizeof(double) * na, e->stream));
    CK(cudaMemsetAsync(reg.p, 0xff, sizeof(int32_t) * na, e->stream));
    DebugOut dbg{e->scratch_a.p, e->scratch_b.p, e->scratch_c.p, e->scratch_d.p, reg.p};
    DevBuf<DevState> st;
    CK(st.ensure(1));
    CK(cudaMemsetAsync(st.p, 0, sizeof(DevState), e->stream));
    // whole list, so every line gets a value irrespective of the owned chunk; the records are scratch here
    // (temporaries, so the live prepass is not disturbed)
    DevBuf<float4> r4, r5; DevBuf<float> r2;
    CK(r4.ensure(na)); CK(r5.ensure(na)); CK(r2.ensure(na));
    K1Table &tab = e->k1_host;
    tab.n = 1;
    K1Layer &row = tab.rows[0];
    row.T = e->last.T; row.P = e->last.P;
    row.lc = layer_consts(e->last.T, e->last.P, e->res);
    row.scale = e->last.scale;
    row.scale_dev = nullptr;
    row.wm = (double)e->last.wm;
    row.gp = e->gp.p;
    row.recA = r4.p; row.recB = r5.p; row.recD = r2.p;
    row.st = st.p;
    row.narrow = 0; row.pad = 0;
    LinesSoA L{e->nu0.p, e->s296.p, e->gair.p, e->gself.p, e->elower.p, e->nair.p, e->delta.p,
               e->has_group ? e->group.p : nullptr};
    k1_prepass<true><<<(unsigned)((na + 255) / 256), 256, 0, e->stream>>>(L, e->idx.p, tab, 0, na, n, e->i_begin, dbg);
    CK(cudaGetLastError());
    if (nu_shift) CK(cudaMemcpyAsync(nu_shift, e->scratch_a.p, sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    if (gamma_l) CK(cudaMemcpyAsync(gamma_l, e->scratch_b.p, sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    if (gamma_d) CK(cudaMemcpyAsync(gamma_d, e->scratch_c.p, sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    if (s_t) CK(cudaMemcpyAsync(s_t, e->scratch_d.p, sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    if (regime) CK(cudaMemcpyAsync(regime, reg.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, e->stream));
    std::vector<int32_t> h_idx(index ? n : 0);
    if (index && n) CK(cudaMemcpyAsync(h_idx.data(), e->idx.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (index) for (int64_t i = 0; i < n; ++i) index[i] = h_idx[i];
    r4.release(); r5.release(); r2.release(); reg.release(); st.release();
    return PRB_OK;
}

// ------------------------------------------------------------------------------------ K2
// Line-range parts (PRB_OPT_SPLIT_TILES): how many work items a (layer, tile) becomes.  A launch of a few waves ends on a
// mostly idle last wave -- 306 equal tiles on 296 resident CTAs take two tile times --; split into S parts of the line
// range the same work is ceil(items S / slots) / S tile times.  Long launches (the batched atmosphere) stay unsplit.
static int pick_parts(const prb_engine *e, int64_t items, int64_t slots) {
    if (!e->split_tiles || items <= 0 || items > 4 * slots) return 1;
    int best = 1;
    double best_t = 1e30;
    for (int s = 1; s <= 8; s *= 2) {
        const double t = (double)((items * s + slots - 1) / slots) / s + 0.015 * s;   // + per-part overhead (search, combine)
        if (t < best_t - 1e-9) { best_t = t; best = s; }
    }
    return best;
}

template <int P>
static cudaError_t launch_k2_t(prb_engine *e, K2Args a) {
    const int tile = K2_CONSUMERS * 32 * P;
    a.n_tiles = (int)((a.n_chunk + tile - 1) / tile);
    if (a.n_tiles == 0) return cudaSuccess;
    const bool staging = a.fuse.enabled && a.fuse.n_dst > 1;
    const size_t smem = K2_SMEM_BYTES<P>(staging);
    int64_t items = (int64_t)a.n_tiles * a.n_layers;
    const int64_t slots = (int64_t)K2_MIN_CTAS * e->prop.multiProcessorCount;
    a.parts = pick_parts(e, items, slots);
    if (a.parts > 1) {
        cudaError_t ce = e->part_sums.ensure((size_t)items * a.parts * tile);
        if (ce == cudaSuccess) ce = e->part_count.ensure((size_t)items);
        if (ce == cudaSuccess) ce = cudaMemsetAsync(e->part_count.p, 0, sizeof(unsigned int) * items, e->stream);
        if (ce != cudaSuccess) return ce;
        a.part_sums = e->part_sums.p;
        a.part_count = e->part_count.p;
        items *= a.parts;
    }
    const int grid = (int)std::min<int64_t>(items, slots);
    const bool far = far_args<P>(e, a);
    if (a.parts > 1) {
        if (far) k2_line_sum_far<(P == 4 ? 4 : 8), true><<<grid, K2_THREADS, smem, e->stream>>>(a);
        else k2_line_sum<P, true><<<grid, K2_THREADS, smem, e->stream>>>(a);
    } else {
        if (far) k2_line_sum_far<(P == 4 ? 4 : 8)><<<grid, K2_THREADS, smem, e->stream>>>(a);
        else k2_line_sum<P><<<grid, K2_THREADS, smem, e->stream>>>(a);
    }
    return cudaGetLastError();
}

static void fill_k2_row(const prb_engine *e, const LayerJob &j, K2Layer &t) {
    const size_t na = (size_t)e->n_alloc;
    t.recA = e->recA.p + na * j.slot;
    t.recB = e->recB.p + na * j.slot;
    t.recD = e->recD.p + na * j.slot;
    t.out = j.out_dev;
    t.inv_scale = 1.0 / j.scale;
    t.l_begin = (int)j.l0;
    t.l_end = (int)j.l1;
    t.wm = (int)j.wm;
    t.pad = 0;
    for (int x = 0; x < K2_MAX_XSC; ++x) t.xsc_w[x] = j.xsc_w[x];
}

// A sub-launch of k2_line_sum<P> over tiles [a.tile_base, a.tile_base + a.n_tiles) of one layer (pipelined upload).
template <int P>
static cudaError_t launch_k2_sub(prb_engine *e, K2Args a, cudaStream_t st) {
    if (a.n_tiles <= 0) return cudaSuccess;
    const bool staging = a.fuse.enabled && a.fuse.n_dst > 1;
    const size_t smem = K2_SMEM_BYTES<P>(staging);
    const int grid = std::min(a.n_tiles, K2_MIN_CTAS * e->prop.multiProcessorCount);
    if (far_args<P>(e, a)) k2_line_sum_far<(P == 4 ? 4 : 8)><<<grid, K2_THREADS, smem, st>>>(a);
    else k2_line_sum<P><<<grid, K2_THREADS, smem, st>>>(a);
    return cudaGetLastError();
}

// Thread-per-point launches: the staged line range of every (layer, tile), precomputed in one parallel pass.
static_assert(KP_TILE == KN_TILE, "k2_point and k2_narrow share the tile size of k2_tile_bounds");
static int tile_bounds(prb_engine *e, K2Args &b) {
    const size_t cnt = (size_t)b.n_layers * b.n_tiles;
    if (e->tile_bounds_buf[e->tile_bounds_next].ensure(cnt) != cudaSuccess)
        return fail(PRB_ERR_CUDA, "tile bounds allocation failed");
    int2 *buf = e->tile_bounds_buf[e->tile_bounds_next].p;
    e->tile_bounds_next ^= 1;                       // two buffers: consecutive launches of one call never share one
    k2_tile_bounds<<<dim3((unsigned)((b.n_tiles + 255) / 256), (unsigned)b.n_layers), 256, 0, e->stream>>>(
        b.layers, b.n_layers, b.idx, b.i_begin, b.n_tiles, KP_TILE, buf);
    CK(cudaGetLastError());
    ++e->extra_launches;
    b.tile_bounds = buf;
    return PRB_OK;
}

// ONE K2 launch for jobs[0..n), which must share a kernel class (all narrow, or all the same ppt) and be sorted
// widest window first.  tab_dev holds the n table rows (fill_k2_row); the launch's tile counter lives in jobs[0]'s
// state block and must be zero (stream-ordered) when the kernel starts.
static void xsc_args(const prb_engine *e, K2Args &a);
static int run_line_sum(prb_engine *e, const LayerJob *jobs, int n, const K2Layer *tab_dev, int out_mode,
                        const K2Fuse *fuse, bool with_xsc = false) {
    if (n <= 0) return PRB_OK;
    K2Args a{};
    if (with_xsc) xsc_args(e, a);
    a.layers = tab_dev;
    a.n_layers = n;
    a.idx = e->idx.p;
    a.i_begin = e->i_begin;
    a.n_chunk = (int)chunk_len(e);
    a.variant = e->k2_variant;
    a.out_mode = out_mode;
    a.st = jobs[0].st_dev;
    if (fuse) a.fuse = *fuse;
    cudaError_t ce;
    if (jobs[0].narrow == 2) {
        a.n_tiles = (a.n_chunk + KP_TILE - 1) / KP_TILE;
        for (int k0 = 0; k0 < n && a.n_tiles > 0; k0 += 65535) {        // grid.y limit
            K2Args b = a;
            b.layers = tab_dev + k0;
            b.n_layers = std::min(n - k0, 65535);
            int rc2 = tile_bounds(e, b);
            if (rc2) return rc2;
            k2_point<<<dim3((unsigned)a.n_tiles, (unsigned)b.n_layers), KP_THREADS, sizeof(KPSmem), e->stream>>>(b);
        }
        ce = cudaGetLastError();
        if (ce != cudaSuccess) return fail(PRB_ERR_CUDA, std::string("k2_point launch failed: ") + cudaGetErrorString(ce));
        return PRB_OK;
    }
    if (jobs[0].narrow) {
        a.n_tiles = (a.n_chunk + KN_TILE - 1) / KN_TILE;
        for (int k0 = 0; k0 < n && a.n_tiles > 0; k0 += 65535) {        // grid.y limit
            K2Args b = a;
            b.layers = tab_dev + k0;
            b.n_layers = std::min(n - k0, 65535);
            int rc2 = tile_bounds(e, b);
            if (rc2) return rc2;
            k2_narrow<<<dim3((unsigned)a.n_tiles, (unsigned)b.n_layers), KN_THREADS, sizeof(KNSmem), e->stream>>>(b);
        }
        ce = cudaGetLastError();
        if (ce != cudaSuccess) return fail(PRB_ERR_CUDA, std::string("k2_narrow launch failed: ") + cudaGetErrorString(ce));
        return PRB_OK;
    }
    switch (jobs[0].ppt) {
        case 2: ce = launch_k2_t<2>(e, a); break;
        case 4: ce = launch_k2_t<4>(e, a); break;
        case 16: ce = launch_k2_t<16>(e, a); break;
        default: ce = launch_k2_t<8>(e, a); break;
    }
    if (ce != cudaSuccess) return fail(PRB_ERR_CUDA, std::string("k2_line_sum launch failed: ") + cudaGetErrorString(ce));
    return PRB_OK;
}

extern "C" int prb_line_sum_dev(prb_engine *e, void *out_dev, int out_mode) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (!e->last.valid) return fail(PRB_ERR_STATE, "prb_line_sum: run prb_layer_prepass first");
    if (!e->seg.empty()) return fail(PRB_ERR_STATE, "prb_line_sum: grouped line list -- use prb_line_sum_groups");
    if (!out_dev) return fail(PRB_ERR_ARG, "prb_line_sum_dev: NULL output");
    if (out_mode != PRB_OUT_F64 && out_mode != PRB_OUT_F32) return fail(PRB_ERR_ARG, "prb_line_sum_dev: bad out_mode");
    CK(cudaSetDevice(e->device));
    LayerJob j = e->last;
    j.out_dev = out_dev;
    // enqueue-only entry point: the table row travels through a small pinned ring (a slot is reused only after
    // the copy that read it has completed), so no host synchronisation is needed here
    if (!e->ring_h) {
        CK(cudaMallocHost((void **)&e->ring_h, sizeof(K2Layer) * RING));
        CK(e->ring_d.ensure(RING));
        for (int k = 0; k < RING; ++k) CK(cudaEventCreateWithFlags(&e->ring_ev[k], cudaEventDisableTiming));
    }
    const int slot = e->ring_next++ % RING;
    CK(cudaEventSynchronize(e->ring_ev[slot]));
    fill_k2_row(e, j, e->ring_h[slot]);
    CK(cudaMemcpyAsync(e->ring_d.p + slot, e->ring_h + slot, sizeof(K2Layer), cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemsetAsync(&j.st_dev->tile_counter, 0, sizeof(unsigned int), e->stream));
    int rc = run_line_sum(e, &j, 1, e->ring_d.p + slot, out_mode, nullptr);
    if (rc) return rc;
    CK(cudaEventRecord(e->ring_ev[slot], e->stream));
    return PRB_OK;
}

extern "C" int prb_line_sum(prb_engine *e, double *out_host) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (!out_host && chunk_len(e) > 0) return fail(PRB_ERR_ARG, "prb_line_sum: NULL output");
    const int64_t nc = e->grid_set ? chunk_len(e) : 0;
    if (!e->last.valid) return fail(PRB_ERR_STATE, "prb_line_sum: run prb_layer_prepass first");
    CK(cudaSetDevice(e->device));
    CK(e->out64.ensure(nc));
    int rc = prb_line_sum_dev(e, e->out64.p, PRB_OUT_F64);
    if (rc) return rc;
    if (nc) CK(cudaMemcpyAsync(out_host, e->out64.p, sizeof(double) * nc, cudaMemcpyDeviceToHost, e->stream));
    rc = check_flags(e, 1);                                     // synchronises
    return rc;
}

// Per-group rows in ONE K2 launch: group g is work-item row g (its own line range, its own output row), all rows share
// the records of the last prepass and the launch's tile counter.  Rows stay on the device (prb_layer_spectra_resident
// reads them there) and are copied to out_host [n_groups][chunk] when it is not NULL.  For a line list uploaded with
// prb_upload_lines (one ascending run with group ids) there is a single row: the sum over the groups.
extern "C" int prb_line_sum_groups(prb_engine *e, double *out_host) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (!e->last.valid) return fail(PRB_ERR_STATE, "prb_line_sum_groups: run prb_layer_prepass first");
    if (e->seg.empty()) return fail(PRB_ERR_STATE, "prb_line_sum_groups: upload the lines with prb_upload_line_groups");
    CK(cudaSetDevice(e->device));
    const int64_t nc = chunk_len(e);
    const int G = e->n_groups;
    CK(e->out64.ensure((size_t)std::max<int64_t>(nc, 1) * G));
    CK(e->k2tab.ensure(G));
    std::vector<LayerJob> jobs(G, e->last);
    std::vector<K2Layer> rows(G);
    for (int g = 0; g < G; ++g) {
        jobs[g].l0 = e->seg[g];
        jobs[g].l1 = e->seg[g] + e->seg_cnt[g];
        jobs[g].out_dev = e->out64.p + (size_t)g * nc;
        fill_k2_row(e, jobs[g], rows[g]);
    }
    CK(cudaMemcpyAsync(e->k2tab.p, rows.data(), sizeof(K2Layer) * G, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemsetAsync(&jobs[0].st_dev->tile_counter, 0, sizeof(unsigned int), e->stream));
    int rc = run_line_sum(e, jobs.data(), G, e->k2tab.p, PRB_OUT_F64, nullptr);
    if (rc) return rc;
    if (out_host && nc) CK(cudaMemcpyAsync(out_host, e->out64.p, sizeof(double) * nc * G, cudaMemcpyDeviceToHost, e->stream));
    rc = check_flags(e, 1);                                     // synchronises (the pageable table copy has left `rows`)
    e->group_rows_valid = rc == PRB_OK;
    return rc;
}

static unsigned stream_grid(const prb_engine *e, int64_t n, int per_thread);
static int ensure_xsc_rows(prb_engine *e);

// absCoef / transmittance / Layer.transmission (pyradClasses.py:581-587, 707-716, 784-787) from rows that are already on
// the device: the per-group cross sections of the last prb_line_sum_groups, weighted by group_weight[g], plus the resident
// xsc tables weighted by xsc_weight[t] (NULL or n_xsc entries).  Host buffers of chunk length in and out, FP64; the
// wavenumber axis is linspace(range_min, range_max, n_total) as in prb_atmosphere.
extern "C" int prb_layer_spectra_resident(prb_engine *e, const double *group_weight, const double *xsc_weight,
                                          double depth_cm, double t_layer, double range_max, const double *radiance_in,
                                          double *abs_coef, double *transmittance, double *radiance_out) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (!e->group_rows_valid) return fail(PRB_ERR_STATE, "prb_layer_spectra_resident: run prb_line_sum_groups first");
    if (!group_weight) return fail(PRB_ERR_ARG, "prb_layer_spectra_resident: NULL weights");
    if (radiance_out && !radiance_in) return fail(PRB_ERR_ARG, "prb_layer_spectra_resident: radiance_out needs radiance_in");
    CK(cudaSetDevice(e->device));
    const int64_t nc = chunk_len(e);
    if (nc == 0) return PRB_OK;
    const int G = e->n_groups, X = xsc_weight ? e->n_xsc : 0;
    int rc = X ? ensure_xsc_rows(e) : PRB_OK;
    if (rc) return rc;
    CK(e->scratch_w.ensure(G + K2_MAX_XSC));
    CK(e->scratch_b.ensure(nc)); CK(e->scratch_c.ensure(nc)); CK(e->scratch_d.ensure(nc));
    CK(cudaMemcpyAsync(e->scratch_w.p, group_weight, sizeof(double) * G, cudaMemcpyHostToDevice, e->stream));
    if (X) CK(cudaMemcpyAsync(e->scratch_w.p + G, xsc_weight, sizeof(double) * X, cudaMemcpyHostToDevice, e->stream));
    if (radiance_out) {
        CK(e->scratch_a.ensure(nc));
        CK(cudaMemcpyAsync(e->scratch_a.p, radiance_in, sizeof(double) * nc, cudaMemcpyHostToDevice, e->stream));
    }
    const double dx = e->n_total > 1 ? (range_max - e->range_min) / (double)(e->n_total - 1) : 0.0;
    k3_layer_stream_rows_f64<<<stream_grid(e, nc, 1), 256, 0, e->stream>>>(
        nc, G, e->out64.p, nc, e->scratch_w.p, X, e->xsc_rows.p, e->xsc_ld, e->scratch_w.p + G, depth_cm, t_layer,
        e->i_begin, e->n_total, e->range_min, dx, range_max, radiance_out ? e->scratch_a.p : nullptr,
        abs_coef ? e->scratch_b.p : nullptr, transmittance ? e->scratch_c.p : nullptr,
        radiance_out ? e->scratch_d.p : nullptr);
    CK(cudaGetLastError());
    if (abs_coef) CK(cudaMemcpyAsync(abs_coef, e->scratch_b.p, sizeof(double) * nc, cudaMemcpyDeviceToHost, e->stream));
    if (transmittance) CK(cudaMemcpyAsync(transmittance, e->scratch_c.p, sizeof(double) * nc, cudaMemcpyDeviceToHost, e->stream));
    if (radiance_out) CK(cudaMemcpyAsync(radiance_out, e->scratch_d.p, sizeof(double) * nc, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return PRB_OK;
}

extern "C" int64_t prb_pair_count(prb_engine *e) {
    if (!e || !e->last.valid) {
        fail(PRB_ERR_STATE, "prb_pair_count: run prb_layer_prepass first");
        return -1;
    }
    if (cudaSetDevice(e->device) != cudaSuccess || e->dev_scal.ensure(8) != cudaSuccess) {
        fail(PRB_ERR_CUDA, "prb_pair_count: device setup failed");
        return -1;
    }
    unsigned long long total = 0;
    cudaMemsetAsync(e->dev_scal.p + 4, 0, sizeof(unsigned long long), e->stream);
    if (e->n_lines > 0)
        k0_pair_count<<<(unsigned)std::min<int64_t>((e->n_lines + 255) / 256, 4096), 256, 0, e->stream>>>(
            e->idx.p, e->n_lines, e->last.wm, e->i_begin, e->i_end - 1, e->dev_scal.p + 4);
    cudaMemcpyAsync(&total, e->dev_scal.p + 4, sizeof total, cudaMemcpyDeviceToHost, e->stream);
    if (cudaStreamSynchronize(e->stream) != cudaSuccess || cudaGetLastError() != cudaSuccess) {
        fail(PRB_ERR_CUDA, "prb_pair_count: device reduction failed");
        return -1;
    }
    return (int64_t)total;
}

// ------------------------------------------------------------------------------------ K3 (host buffers)
static unsigned stream_grid(const prb_engine *e, int64_t n, int per_thread = 1);
static unsigned stream_grid(const prb_engine *e, int64_t n, int per_thread) {
    const int64_t blocks = (n / per_thread + 255) / 256;
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)e->prop.multiProcessorCount * 16));
}

extern "C" int prb_layer_stream(prb_engine *e, int64_t n, int32_t n_mol, const double *sigma, const double *weight,
                                double depth_cm, double t_layer, double x0, double dx, double x_last,
                                const double *radiance_in, double *abs_coef, double *transmittance,
                                double *radiance_out) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n < 0 || n_mol < 0) return fail(PRB_ERR_ARG, "prb_layer_stream: negative size");
    if (n_mol > 0 && (!sigma || !weight)) return fail(PRB_ERR_ARG, "prb_layer_stream: NULL sigma/weight");
    if (radiance_out && !radiance_in) return fail(PRB_ERR_ARG, "prb_layer_stream: radiance_out needs radiance_in");
    if (n == 0) return PRB_OK;
    CK(cudaSetDevice(e->device));
    CK(e->scratch_a.ensure((size_t)n * std::max(n_mol, 1)));
    CK(e->scratch_w.ensure(std::max(n_mol, 1)));
    CK(e->scratch_b.ensure(n)); CK(e->scratch_c.ensure(n)); CK(e->scratch_d.ensure(n));
    DevBuf<double> rin;
    if (n_mol) {
        CK(cudaMemcpyAsync(e->scratch_a.p, sigma, sizeof(double) * n * n_mol, cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemcpyAsync(e->scratch_w.p, weight, sizeof(double) * n_mol, cudaMemcpyHostToDevice, e->stream));
    }
    if (radiance_out) {
        CK(rin.ensure(n));
        CK(cudaMemcpyAsync(rin.p, radiance_in, sizeof(double) * n, cudaMemcpyHostToDevice, e->stream));
    }
    k3_layer_stream_f64<<<stream_grid(e, n), 256, 0, e->stream>>>(
        n, n_mol, e->scratch_a.p, e->scratch_w.p, depth_cm, t_layer, x0, dx, x_last, radiance_out ? rin.p : nullptr,
        abs_coef ? e->scratch_b.p : nullptr, transmittance ? e->scratch_c.p : nullptr,
        radiance_out ? e->scratch_d.p : nullptr);
    CK(cudaGetLastError());
    if (abs_coef) CK(cudaMemcpyAsync(abs_coef, e->scratch_b.p, sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    if (transmittance) CK(cudaMemcpyAsync(transmittance, e->scratch_c.p, sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    if (radiance_out) CK(cudaMemcpyAsync(radiance_out, e->scratch_d.p, sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    rin.release();
    return PRB_OK;
}

extern "C" int prb_planck(prb_engine *e, int64_t n, double x0, double dx, double x_last, double temp, double *out) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n < 0 || (n > 0 && !out)) return fail(PRB_ERR_ARG, "prb_planck: bad arguments");
    if (n == 0) return PRB_OK;
    CK(cudaSetDevice(e->device));
    CK(e->scratch_b.ensure(n));
    k3_planck_f64<<<stream_grid(e, n), 256, 0, e->stream>>>(n, x0, dx, x_last, temp, e->scratch_b.p);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, e->scratch_b.p, sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return PRB_OK;
}

extern "C" int prb_xsc_place(prb_engine *e, int64_t n_out, int64_t dst0, int64_t src0, int64_t count, int interp,
                             double ax0, double adelta, int64_t n_file, const double *file_x, const double *file_y,
                             double *out) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n_out < 0 || count < 0 || n_file < 1 || !file_y || (interp && !file_x) || (n_out > 0 && !out))
        return fail(PRB_ERR_ARG, "prb_xsc_place: bad arguments");
    if (n_out == 0) return PRB_OK;
    CK(cudaSetDevice(e->device));
    CK(e->scratch_a.ensure(n_file)); CK(e->scratch_c.ensure(n_file)); CK(e->scratch_b.ensure(n_out));
    if (interp) CK(cudaMemcpyAsync(e->scratch_a.p, file_x, sizeof(double) * n_file, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemcpyAsync(e->scratch_c.p, file_y, sizeof(double) * n_file, cudaMemcpyHostToDevice, e->stream));
    k3_xsc_place<<<stream_grid(e, n_out), 256, 0, e->stream>>>(n_out, dst0, src0, count, interp, ax0, adelta, n_file,
                                                              e->scratch_a.p, e->scratch_c.p, e->scratch_b.p, 0);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, e->scratch_b.p, sizeof(double) * n_out, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return PRB_OK;
}

// ------------------------------------------------------------------------------------ resident xsc tables
// An xsc molecule's cross section does not depend on the layer (the table IS the spectrum at its own T and P,
// pyradClasses.py:466-505), so the table is kept on the device with its placement plan and resampled onto the owned grid
// chunk once per grid (k3_xsc_place: np.interp arithmetic + aligned placement); every layer's line sum then picks up
// sigma_t * conc_t P / 1e4 / kB / T in K2's epilogue (k2_add_xsc) -- no separate pass over k, no host round trip.
extern "C" int prb_xsc_resident(prb_engine *e, int32_t slot, int64_t n_out, int64_t dst0, int64_t src0, int64_t count,
                                int interp, double ax0, double adelta, int64_t n_file, const double *file_x,
                                const double *file_y) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (slot < 0 || slot >= K2_MAX_XSC || slot > e->n_xsc)
        return fail(PRB_ERR_ARG, "prb_xsc_resident: slot must be an existing table or the next free one (at most 8 tables)");
    if (n_out < 0 || count < 0 || n_file < 1 || !file_y || (interp && !file_x))
        return fail(PRB_ERR_ARG, "prb_xsc_resident: bad arguments");
    CK(cudaSetDevice(e->device));
    XscTable &t = e->xsc[slot];
    t.n_out = n_out; t.dst0 = dst0; t.src0 = src0; t.count = count; t.interp = interp; t.ax0 = ax0; t.adelta = adelta;
    t.n_file = n_file;
    CK(t.fx.ensure(n_file));
    CK(t.fy.ensure(n_file));
    if (interp) CK(cudaMemcpyAsync(t.fx.p, file_x, sizeof(double) * n_file, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemcpyAsync(t.fy.p, file_y, sizeof(double) * n_file, cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));                       // the caller's arrays are free again
    if (slot == e->n_xsc) ++e->n_xsc;
    e->xsc_rows_valid = false;
    return PRB_OK;
}

extern "C" int prb_xsc_clear(prb_engine *e) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    e->n_xsc = 0;
    e->xsc_rows_valid = false;
    e->xsc_conc.clear();
    e->xsc_conc_layers = 0;
    return PRB_OK;
}

// Per-layer line ranges (the reference's gatherData(effectiveRangeMin, effectiveRangeMax) filter, strict on both sides).
extern "C" int prb_set_layer_line_range(prb_engine *e, int32_t n_layers, const double *nu_lo, const double *nu_hi) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n_layers < 0 || (n_layers > 0 && (!nu_lo || !nu_hi)))
        return fail(PRB_ERR_ARG, "prb_set_layer_line_range: bad arguments");
    e->line_lo.assign(nu_lo, nu_lo + n_layers);
    e->line_hi.assign(nu_hi, nu_hi + n_layers);
    return PRB_OK;
}

extern "C" int prb_set_xsc_conc(prb_engine *e, int32_t n_layers, int32_t n_xsc, const double *conc) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n_layers < 0 || n_xsc != e->n_xsc || (n_layers > 0 && n_xsc > 0 && !conc))
        return fail(PRB_ERR_ARG, "prb_set_xsc_conc: n_xsc must equal the number of resident tables");
    e->xsc_conc.assign(conc, conc + (size_t)n_layers * n_xsc);
    e->xsc_conc_layers = n_layers;
    return PRB_OK;
}

// The resident tables resampled onto the owned chunk (rebuilt when the grid or a table changed); enqueue only.
static int ensure_xsc_rows(prb_engine *e) {
    if (e->n_xsc == 0) return PRB_OK;
    if (e->xsc_rows_valid && e->xsc_sig[0] == e->i_begin && e->xsc_sig[1] == e->i_end && e->xsc_sig[2] == e->n_total)
        return PRB_OK;
    const int64_t nc = chunk_len(e);
    e->xsc_ld = (nc + 3) & ~int64_t(3);
    CK(e->xsc_rows.ensure((size_t)std::max<int64_t>(e->xsc_ld, 1) * e->n_xsc));
    for (int t = 0; t < e->n_xsc; ++t) {
        const XscTable &x = e->xsc[t];
        if (x.n_out != e->n_total)
            return fail(PRB_ERR_ARG, "resident xsc table was planned for a different grid length (prb_xsc_resident n_out)");
        if (nc > 0)
            k3_xsc_place<<<stream_grid(e, nc), 256, 0, e->stream>>>(nc, x.dst0, x.src0, x.count, x.interp, x.ax0, x.adelta,
                                                                    x.n_file, x.fx.p, x.fy.p,
                                                                    e->xsc_rows.p + (size_t)t * e->xsc_ld, e->i_begin);
        CK(cudaGetLastError());
        ++e->xsc_build_launches;
    }
    e->xsc_rows_valid = true;
    e->xsc_sig[0] = e->i_begin; e->xsc_sig[1] = e->i_end; e->xsc_sig[2] = e->n_total;
    return PRB_OK;
}

extern "C" int prb_set_continuum(prb_engine *e, int64_t n_table, const double *table_nu, const double *c_self,
                                 const double *c_foreign, const double *t_exp, double t_ref, double p_ref,
                                 int32_t n_layers, const double *mole_fraction) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n_table == 0) {
        e->cont_tab.clear();
        e->cont_x.clear();
        return PRB_OK;
    }
    if (n_table < 2 || !table_nu || !c_self || !c_foreign || !t_exp)
        return fail(PRB_ERR_ARG, "prb_set_continuum: need n_table = 0, or n_table >= 2 and all four tables");
    for (int64_t i = 0; i < n_table; ++i) {
        if (!std::isfinite(table_nu[i]) || (i > 0 && !(table_nu[i] > table_nu[i - 1])))
            return fail(PRB_ERR_ARG, "prb_set_continuum: table_nu must be finite and strictly ascending");
        if (!(std::isfinite(c_self[i]) && c_self[i] >= 0 && std::isfinite(c_foreign[i]) && c_foreign[i] >= 0))
            return fail(PRB_ERR_ARG, "prb_set_continuum: every c_self and c_foreign must be finite and >= 0");
        if (!std::isfinite(t_exp[i])) return fail(PRB_ERR_ARG, "prb_set_continuum: every t_exp must be finite");
    }
    if (!(std::isfinite(t_ref) && t_ref > 0 && std::isfinite(p_ref) && p_ref > 0))
        return fail(PRB_ERR_ARG, "prb_set_continuum: t_ref and p_ref must be finite and > 0");
    if (n_layers < 1 || !mole_fraction) return fail(PRB_ERR_ARG, "prb_set_continuum: need n_layers >= 1 and mole_fraction");
    for (int l = 0; l < n_layers; ++l)
        if (!(mole_fraction[l] >= 0 && mole_fraction[l] <= 1))
            return fail(PRB_ERR_ARG, "prb_set_continuum: every mole fraction must lie in [0, 1]");
    e->cont_tab.assign(table_nu, table_nu + n_table);
    for (const double *p : {c_self, c_foreign, t_exp}) e->cont_tab.insert(e->cont_tab.end(), p, p + n_table);
    e->cont_t_ref = t_ref;
    e->cont_p_ref = p_ref;
    e->cont_x.assign(mole_fraction, mole_fraction + n_layers);
    return PRB_OK;
}

// The continuum table resampled onto the owned chunk (k3_continuum_rows; rebuilt when the grid or the table changed,
// so a caller that sets and clears the same table around every column resamples it once), after kmat_ld is set for
// the call.  Enqueue only; *launches counts a rebuild.
static int ensure_continuum_rows(prb_engine *e, double range_max, int *launches) {
    const int64_t nc = chunk_len(e);
    const double sig[5] = {(double)e->i_begin, (double)e->i_end, (double)e->n_total, e->range_min, range_max};
    if (e->cont_rows_tab == e->cont_tab && std::equal(sig, sig + 5, e->cont_sig)) return PRB_OK;
    const int64_t n_tab = (int64_t)e->cont_tab.size() / 4;
    CK(e->cont_tab_dev.ensure(e->cont_tab.size()));
    CK(cudaMemcpyAsync(e->cont_tab_dev.p, e->cont_tab.data(), sizeof(double) * e->cont_tab.size(), cudaMemcpyHostToDevice,
                       e->stream));
    CK(e->cont_rows.ensure((size_t)3 * std::max<int64_t>(e->kmat_ld, 4)));
    const double dx = e->n_total > 1 ? (range_max - e->range_min) / (double)(e->n_total - 1) : 0.0;
    k3_continuum_rows<<<stream_grid(e, e->kmat_ld), 256, 0, e->stream>>>(nc, e->kmat_ld, e->i_begin, e->n_total,
                                                                        e->range_min, dx, range_max, e->cont_tab_dev.p,
                                                                        n_tab, e->cont_rows.p);
    CK(cudaGetLastError());
    ++*launches;
    e->cont_rows_tab = e->cont_tab;
    std::copy(sig, sig + 5, e->cont_sig);
    return PRB_OK;
}

static void xsc_args(const prb_engine *e, K2Args &a) {
    a.n_xsc = e->n_xsc;
    a.xsc_sigma = e->xsc_rows.p;
    a.xsc_ld = e->xsc_ld;
}

// ------------------------------------------------------------------------------------ atmosphere
static float *peer_slot(const prb_engine *e, int dst, int parity, int field, int src_rank) {
    const PeerState &ps = e->peer;
    return reinterpret_cast<float *>(ps.base[dst] + PEER_HEADER) +
           ((size_t)(parity * 2 + field) * ps.world + src_rank) * (size_t)ps.ld;
}

// Pipelined upload of a gas cell (prb_gas_cell_host): the line columns arrive in S pieces on a copy stream, piece s
// completes event ev[s]; sub-launch s of K2 covers tiles [tile_lo[s], tile_hi[s]) -- one full wave of CTAs -- and
// needs lines [line_lo[s], line_hi[s]); K0/K1 for the lines of piece s = [line_hi[s-1], line_hi[s]).
struct UploadPipe {
    int S = 0;
    std::vector<int64_t> line_lo, line_hi;
    std::vector<int> tile_lo, tile_hi;
    std::vector<cudaEvent_t> ev;                 // piece s has landed
    std::vector<cudaEvent_t> ev_k1;              // K1 of piece s is done (the two compute streams alternate)
    cudaStream_t stream2 = nullptr;
    std::function<int(int)> enqueue_piece;       // puts the copies of piece s on the copy stream and records ev[s]
    const unsigned long long *smax_bits_dev = nullptr;   // max|S296| as computed on the device
    double *scale_dev = nullptr;
};

static int atmosphere_impl(prb_engine *e, int32_t n_layers, int32_t n_groups, const double *depth_cm,
                           const double *t_layer, const double *p_layer, const double *conc, const double *molmass,
                           const double *q_t, const double *q_296, const int64_t *window_len, double t_surface,
                           double range_max, const UploadPipe *pipe) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (!e->grid_set && !pipe) return fail(PRB_ERR_STATE, "prb_atmosphere: set the grid first");
    if (!e->seg.empty() && !pipe)
        return fail(PRB_ERR_STATE, "prb_atmosphere: the line list was uploaded in groups (prb_upload_line_groups); the column "
                                   "path needs one ascending list with group ids (prb_upload_lines)");
    if (n_layers < 1 || n_groups != e->n_groups) return fail(PRB_ERR_ARG, "prb_atmosphere: bad n_layers / n_groups");
    if (!depth_cm || !t_layer || !p_layer || !conc || !molmass || !q_t || !q_296 || !window_len)
        return fail(PRB_ERR_ARG, "prb_atmosphere: NULL array");
    CK(cudaSetDevice(e->device));
    const int64_t nc = chunk_len(e);
    int64_t wmax = 0;
    for (int l = 0; l < n_layers; ++l) {
        if (window_len[l] < 1) return fail(PRB_ERR_ARG, "prb_atmosphere: window_len must be >= 1");
        wmax = std::max<int64_t>(wmax, window_len[l] - 2);
    }
    int rc = check_segment(e, wmax);
    if (rc) return rc;
    PeerState &ps = e->peer;
    if (ps.connected && nc > ps.ld) return fail(PRB_ERR_ARG, "prb_atmosphere: owned chunk exceeds the peer gather slot");
    if (e->host_rad_dev && nc > e->host_result_len)
        return fail(PRB_ERR_ARG, "prb_atmosphere: owned chunk exceeds the host result buffers (prb_set_result_host)");
    if (e->n_xsc > 0 && e->xsc_conc_layers != n_layers)
        return fail(PRB_ERR_ARG, "prb_atmosphere: resident xsc tables need their mole fractions for these layers "
                                 "(prb_set_xsc_conc with the same n_layers), or prb_xsc_clear");
    if (!e->line_lo.empty() && (int)e->line_lo.size() != n_layers)
        return fail(PRB_ERR_ARG, "prb_atmosphere: the per-layer line ranges were set for another number of layers "
                                 "(prb_set_layer_line_range with the same n_layers, or with 0 to clear)");
    const bool continuum = !e->cont_tab.empty();
    if (continuum && (int)e->cont_x.size() != n_layers)
        return fail(PRB_ERR_ARG, "prb_atmosphere: the continuum's mole fractions were set for another number of layers "
                                 "(prb_set_continuum with the same n_layers, or with n_table = 0 to clear)");
    const int xsc_before = e->xsc_build_launches;
    if ((rc = ensure_xsc_rows(e))) return rc;
    const int xsc_launches = e->xsc_build_launches - xsc_before;   // table resamplings this call had to enqueue

    // Everything small the kernels of this call read -- status blocks (zeroed: flags + tile counters), per-(layer,
    // group) params, fold constants, the K2 launch table (K1's is a kernel parameter) -- is built in ONE pinned block and uploaded with
    // ONE copy, so a step is a copy plus its kernel launches.
    const int n_rows = pipe ? std::max(pipe->S, 1) : n_layers;      // status blocks / K2 table rows (one per launch item)
    const size_t off_st = 0;
    const size_t off_gp = off_st + sizeof(DevState) * n_rows;
    const size_t off_fold = off_gp + sizeof(GroupParams) * (size_t)n_layers * n_groups;
    const size_t off_k2 = (off_fold + sizeof(FoldLayer) * n_layers + 15) & ~size_t(15);
    const size_t blk_bytes = off_k2 + sizeof(K2Layer) * n_rows;
    if (blk_bytes > e->blk_cap) {
        if (e->blk_h) cudaFreeHost(e->blk_h);
        e->blk_h = nullptr;
        e->blk_cap = 0;
        CK(cudaMallocHost((void **)&e->blk_h, blk_bytes));
        e->blk_cap = blk_bytes;
    }
    CK(e->blk_d.ensure(blk_bytes));
    memset(e->blk_h, 0, blk_bytes);
    DevState *st_dev = reinterpret_cast<DevState *>(e->blk_d.p + off_st);
    GroupParams *gp_dev = reinterpret_cast<GroupParams *>(e->blk_d.p + off_gp);
    FoldLayer *fold_dev = reinterpret_cast<FoldLayer *>(e->blk_d.p + off_fold);
    K2Layer *k2_dev = reinterpret_cast<K2Layer *>(e->blk_d.p + off_k2);
    GroupParams *h = reinterpret_cast<GroupParams *>(e->blk_h + off_gp);
    FoldLayer *hf = reinterpret_cast<FoldLayer *>(e->blk_h + off_fold);
    K2Layer *k2rows = reinterpret_cast<K2Layer *>(e->blk_h + off_k2);

    // per-(layer, group) params: weight = conc * P / 1e4 / kB / T  (absCoef, pyradClasses.py:581-583)
    std::vector<LayerJob> jobs(n_layers);
    const double c2 = 100 * hPlanck * cLight / kBoltz;
    e->kmat_ld = (nc + 3) & ~int64_t(3);
    CK(e->kmat.ensure((size_t)e->kmat_ld * n_layers));
    CK(e->rad.ensure(e->kmat_ld));
    CK(e->trans.ensure(e->kmat_ld));
    std::vector<double> w(n_groups);
    double pipe_w_max = 1.0;
    for (int l = 0; l < n_layers; ++l) {
        for (int g = 0; g < n_groups; ++g)
            w[g] = conc[(size_t)l * n_groups + g] * p_layer[l] / 1E4 / kBoltz / t_layer[l];
        double w_max = 0;
        build_group_params(n_groups, t_layer[l], conc + (size_t)l * n_groups, molmass, q_t + (size_t)l * n_groups,
                           q_296, w.data(), h + (size_t)l * n_groups, &w_max);
        hf[l].neg_depth_log2e = (float)(-depth_cm[l] * 1.4426950408889634);
        hf[l].c2_over_t = (float)(c2 / t_layer[l]);
        if (pipe) {                                             // the grid indices are not on the host yet
            LayerJob &j = jobs[l];
            j.T = t_layer[l]; j.P = p_layer[l]; j.W = window_len[l];
            j.scale = 1.0;                                      // placeholder: the device computes it (k0_pick_scale)
            j.scale_dev = pipe->scale_dev;
            pipe_w_max = w_max;
            j.wm = std::max<int64_t>(window_len[l] - 2, 0);
            j.l0 = 0; j.l1 = e->n_lines;
            j.narrow = 0;
            j.ppt = pick_ppt(e, j.wm);
            j.valid = true;
        } else {
            jobs[l] = plan_job(e, t_layer[l], p_layer[l], window_len[l], pick_scale(e->s_max, w_max));
        }
        for (int x = 0; x < e->n_xsc; ++x)                      // absCoef of an xsc molecule, same factor (:581-583)
            jobs[l].xsc_w[x] = e->xsc_conc[(size_t)l * e->n_xsc + x] * p_layer[l] / 1E4 / kBoltz / t_layer[l];
        if (!e->line_lo.empty()) {
            jobs[l].filter = true;
            jobs[l].nu_lo = e->line_lo[l];
            jobs[l].nu_hi = e->line_hi[l];
        }
        jobs[l].gp_dev = gp_dev + (size_t)l * n_groups;
        jobs[l].st_dev = st_dev + l;
        jobs[l].out_dev = e->kmat.p + (size_t)l * e->kmat_ld;
    }
    if (e->atm_layers != n_layers) {
        CK(cudaMemsetAsync(e->kmat.p, 0, sizeof(float) * e->kmat_ld * n_layers, e->stream));
        e->atm_layers = n_layers;
    }
    e->atm_depth.assign(depth_cm, depth_cm + n_layers);
    e->atm_t.assign(t_layer, t_layer + n_layers);
    e->atm_t_surface = t_surface;
    e->atm_range_max = range_max;
    e->atm_nu_interp_min = 1e30f;                                // per-point Planck unless k3_fold_tma runs below

    // Launch plan.  Layers are processed widest window first, in batches of `slots` layers whose records are
    // resident together (36 B per line per layer): ONE K1 launch per batch, then ONE K2 launch per kernel class
    // of the batch, each walking all its (layer, tile) items from one dynamic counter -- a handful of launch
    // tails per atmosphere instead of one per layer, which is what strong scaling over small chunks needs.
    std::stable_sort(jobs.begin(), jobs.end(), [](const LayerJob &x, const LayerJob &y) { return x.wm > y.wm; });
    int64_t slots = 1;
    if (e->batch_layers && n_layers > 1 && e->rec_slots >= n_layers && e->rec_budget_mb == 0) {
        slots = n_layers;                                       // the records of every layer are already resident
    } else if (e->batch_layers && n_layers > 1) {
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));                  // (a driver query: only when the batch has to be sized)
        const size_t per_layer = (size_t)36 * (size_t)std::max<int64_t>(e->n_alloc, 1);
        const size_t have = (size_t)e->rec_slots * per_layer;               // already allocated records count as free
        const size_t budget = e->rec_budget_mb > 0 ? (size_t)e->rec_budget_mb << 20 : (free_b + have) / 4;
        slots = std::max<int64_t>(1, std::min<int64_t>(n_layers, (int64_t)(budget / per_layer)));
    }
    if ((rc = ensure_records(e, slots))) return rc;

    // destinations of the finished spectra
    unsigned int epoch = 0;
    K3Dst dst{};
    if (ps.connected) {
        epoch = ++ps.epoch;
        dst.n = ps.world;
        for (int d = 0; d < ps.world; ++d) {
            dst.rad[d] = peer_slot(e, d, epoch & 1, 0, ps.rank);
            dst.trans[d] = peer_slot(e, d, epoch & 1, 1, ps.rank);
        }
        e->res_rad = dst.rad[ps.rank];
        e->res_trans = dst.trans[ps.rank];
    } else {
        dst.n = 1;
        dst.rad[0] = e->rad.p;
        dst.trans[0] = e->trans.p;
        e->res_rad = e->rad.p;
        e->res_trans = e->trans.p;
    }
    if (e->host_rad_dev) {                                      // zero-copy result delivery (prb_set_result_host)
        dst.rad[dst.n] = e->host_rad_dev;
        dst.trans[dst.n] = e->host_trans_dev;
        ++dst.n;
    }
    const double dx = e->n_total > 1 ? (range_max - e->range_min) / (double)(e->n_total - 1) : 0.0;
    // a continuum is added to the k matrix between K2 and the fold, so it needs the separate fold
    const bool fused = n_layers == 1 && e->fuse_single && !jobs[0].narrow && k2_classed(e) && !continuum;
    K2Fuse fuse{};
    if (fused) {
        fuse.enabled = 1;
        fuse.n_dst = dst.n;
        fuse.neg_depth_log2e = (float)(-depth_cm[0] * 1.4426950408889634);
        fuse.c2_over_t = (float)(c2 / t_layer[0]);
        fuse.c2_over_tsurf = (float)(c2 / t_surface);
        fuse.n_total = e->n_total;
        fuse.x0 = e->range_min; fuse.dx = dx; fuse.x_last = range_max;
        for (int d = 0; d < dst.n; ++d) { fuse.rad[d] = dst.rad[d]; fuse.trans[d] = dst.trans[d]; }
    }

    const int n_batches = (int)((n_layers + slots - 1) / slots);
    const size_t n_ev = (size_t)3 * n_batches + 2;
    if (e->timing) {
        while (e->ev.size() < n_ev) {
            cudaEvent_t x;
            CK(cudaEventCreate(&x));
            e->ev.push_back(x);
        }
    }
    for (int k = 0; k < n_layers; ++k) {
        jobs[k].slot = (int)(k % slots);
        fill_k2_row(e, jobs[k], k2rows[k]);
    }
    if (pipe) {
        for (int sidx = 0; sidx < pipe->S; ++sidx) {            // one K2 table row per sub-launch: its own line range
            k2rows[sidx] = k2rows[0];
            k2rows[sidx].l_begin = (int)pipe->line_lo[sidx];
            k2rows[sidx].l_end = (int)pipe->line_hi[sidx];
        }
    }
    CK(cudaMemcpyAsync(e->blk_d.p, e->blk_h, blk_bytes, cudaMemcpyHostToDevice, e->stream));
    int launches = xsc_launches;
    e->extra_launches = 0;
    if (pipe) {
        if (!fused) return fail(PRB_ERR_STATE, "pipelined upload needs the fused single-layer path");
        const int64_t n = e->n_lines, na = e->n_alloc;
        // the scale of the records, on the device: into K1's scale word and (inverted) the K2 table rows
        static_assert(sizeof(K2Layer) % sizeof(double) == 0, "K2Layer rows are addressed in doubles");
        k0_pick_scale<<<1, 32, 0, e->stream>>>(pipe->smax_bits_dev, pipe_w_max, pipe->scale_dev,
                                              &k2_dev[0].inv_scale, pipe->S, (int)(sizeof(K2Layer) / sizeof(double)));
        CK(cudaGetLastError());
        CK(cudaEventRecord(pipe->ev_k1[pipe->S], e->stream));     // "tables ready" for the second stream
        CK(cudaStreamWaitEvent(pipe->stream2, pipe->ev_k1[pipe->S], 0));
        // Sub-launches alternate between two streams: while the tail of wave s drains (its CTAs retire one by one, its
        // bulk stores to the host / peers complete), K0/K1/K2 of wave s+1 already run on the freed SMs.
        for (int sidx = 0; sidx < pipe->S; ++sidx) {
            // keep the copy stream one piece ahead of the launches (the host enqueues both; neither should wait for it)
            if (sidx + 1 < pipe->S && (rc = pipe->enqueue_piece(sidx + 1))) return rc;
            cudaStream_t st = (sidx & 1) ? pipe->stream2 : e->stream;
            CK(cudaStreamWaitEvent(st, pipe->ev[sidx], 0));
            if (sidx) CK(cudaStreamWaitEvent(st, pipe->ev_k1[sidx - 1], 0));   // records of the earlier pieces
            // K0 + K1 for the lines this piece brought (the last piece also writes the padding records)
            const int64_t a = sidx ? pipe->line_hi[sidx - 1] : 0;
            const int64_t b = sidx == pipe->S - 1 ? na : pipe->line_hi[sidx];
            if (b > a) {
                k0_line_index<<<(unsigned)((b - a + 255) / 256), 256, 0, st>>>(e->nu0.p, n, a, b, e->range_min, e->res, e->idx.p);
                CK(cudaGetLastError());
                LayerJob jj = jobs[0];
                jj.l0 = a;
                jj.l1 = std::min<int64_t>(b, n);
                K1Table &tab = e->k1_host;
                tab.n = 1;
                tab.pad = 0;
                fill_k1_row(e, jj, tab.rows[0]);
                LinesSoA Ls{e->nu0.p, e->s296.p, e->gair.p, e->gself.p, e->elower.p, e->nair.p, e->delta.p,
                            e->has_group ? e->group.p : nullptr};
                k1_prepass<false><<<(unsigned)((b - a + 255) / 256), 256, 0, st>>>(Ls, e->idx.p, tab, a, b, n, e->i_begin, DebugOut{});
                CK(cudaGetLastError());
                launches += 2;
            }
            CK(cudaEventRecord(pipe->ev_k1[sidx], st));
            // K2 over this piece's wave of tiles
            K2Args ka{};
            ka.layers = k2_dev + sidx;
            ka.n_layers = 1;
            ka.idx = e->idx.p;
            ka.i_begin = e->i_begin;
            ka.n_chunk = (int)nc;
            ka.variant = e->k2_variant;
            ka.out_mode = PRB_OUT_F32;
            ka.st = st_dev + sidx;
            ka.fuse = fuse;
            xsc_args(e, ka);
            ka.tile_base = pipe->tile_lo[sidx];
            ka.n_tiles = pipe->tile_hi[sidx] - pipe->tile_lo[sidx];
            cudaError_t ce;
            switch (jobs[0].ppt) {
                case 2: ce = launch_k2_sub<2>(e, ka, st); break;
                case 4: ce = launch_k2_sub<4>(e, ka, st); break;
                case 16: ce = launch_k2_sub<16>(e, ka, st); break;
                default: ce = launch_k2_sub<8>(e, ka, st); break;
            }
            if (ce != cudaSuccess) return fail(PRB_ERR_CUDA, std::string("k2_line_sum sub-launch failed: ") + cudaGetErrorString(ce));
            ++launches;
        }
        CK(cudaEventRecord(pipe->ev_k1[pipe->S], pipe->stream2));  // join: everything after this sees both streams' work
        CK(cudaStreamWaitEvent(e->stream, pipe->ev_k1[pipe->S], 0));
    }
    for (int bi = 0; bi < (pipe ? 0 : n_batches); ++bi) {
        const int b0 = (int)(bi * slots), b1 = (int)std::min<int64_t>(n_layers, b0 + slots);
        if (e->timing) CK(cudaEventRecord(e->ev[3 * bi], e->stream));
        rc = run_prepass(e, jobs.data() + b0, b1 - b0, DebugOut{}, &launches);
        if (rc) return rc;
        if (e->timing) CK(cudaEventRecord(e->ev[3 * bi + 1], e->stream));
        for (int c0 = b0; c0 < b1;) {                            // runs of one kernel class (sorted by window)
            int c1 = c0 + 1;
            while (c1 < b1 && jobs[c1].narrow == jobs[c0].narrow && (jobs[c0].narrow || jobs[c1].ppt == jobs[c0].ppt)) ++c1;
            rc = run_line_sum(e, jobs.data() + c0, c1 - c0, k2_dev + c0, PRB_OUT_F32, fused ? &fuse : nullptr, true);
            if (rc) return rc;
            ++launches;
            c0 = c1;
        }
        if (e->timing) CK(cudaEventRecord(e->ev[3 * bi + 2], e->stream));
    }
    if (e->timing) CK(cudaEventRecord(e->ev[3 * n_batches], e->stream));
    if (continuum && nc > 0) {
        // the continuum on the finished k matrix: the layers with x > 0, their constants formed in FP64
        if ((rc = ensure_continuum_rows(e, range_max, &launches))) return rc;
        std::vector<ContLayer> cl;
        for (int l = 0; l < n_layers; ++l) {
            const double x = e->cont_x[l];
            if (!(x > 0)) continue;
            const double n_rho = x * p_layer[l] / 1E4 / kBoltz / t_layer[l] * (p_layer[l] / e->cont_p_ref) *
                                 (e->cont_t_ref / t_layer[l]);
            cl.push_back(ContLayer{(float)(n_rho * x), (float)(n_rho * (1 - x)), (float)std::log2(e->cont_t_ref / t_layer[l]),
                                   (float)(c2 / (2 * t_layer[l])), l, 0});
        }
        if (!cl.empty()) {
            CK(e->cont_layers.ensure(cl.size()));
            CK(cudaMemcpyAsync(e->cont_layers.p, cl.data(), sizeof(ContLayer) * cl.size(), cudaMemcpyHostToDevice, e->stream));
            k3_continuum_add<<<stream_grid(e, e->kmat_ld, 4), 256, 0, e->stream>>>(
                e->kmat.p, e->kmat_ld, e->cont_layers.p, (int)cl.size(), e->cont_rows.p, e->i_begin, e->n_total,
                e->range_min, dx, range_max);
            CK(cudaGetLastError());
            ++launches;
        }
    }
    if (nc > 0 && !fused) {
        if (e->k3_tma && n_layers >= K3T_LAYERS) {
            const int64_t n_strips = (nc + K3T_STRIP - 1) / K3T_STRIP;
            const int grid = (int)std::min<int64_t>(n_strips, K3T_MINB * (int64_t)e->prop.multiProcessorCount);
            // linear interpolation of B over 3 grid steps: relative error <= (3 dx)^2 / 8 * max(6 / nu^2, (c2/T)^2);
            // keep it below 1e-7, and stay where x = c2 nu / T >= 0.25 for every layer (no expm1 branch)
            double t_max = t_surface, t_min = t_surface;
            for (int l = 0; l < n_layers; ++l) { t_max = std::max(t_max, t_layer[l]); t_min = std::min(t_min, t_layer[l]); }
            double nu_min = std::max(3 * dx * std::sqrt(6.0 / 8e-7), 0.26 * t_max / c2);
            if ((3 * dx) * (3 * dx) / 8 * (c2 / t_min) * (c2 / t_min) > 1e-7) nu_min = 1e30;      // grid too coarse: never
            e->atm_nu_interp_min = (float)nu_min;
            k3_fold_tma<<<grid, K3T_THREADS, sizeof(K3TSmem), e->stream>>>(e->kmat.p, e->kmat_ld, n_layers, fold_dev, nc,
                                                                          e->i_begin, e->n_total, e->range_min, dx, range_max,
                                                                          (float)(c2 / t_surface), (float)nu_min, dst);
        } else {
            k3_fold_f32<<<stream_grid(e, nc, 4), 256, 0, e->stream>>>(e->kmat.p, e->kmat_ld, n_layers, fold_dev, nc,
                                                                     e->i_begin, e->n_total, e->range_min, dx, range_max,
                                                                     (float)(c2 / t_surface), dst);
        }
        CK(cudaGetLastError());
        ++launches;
    }
    if (e->timing) CK(cudaEventRecord(e->ev[3 * n_batches + 1], e->stream));
    if (ps.connected) {
        PeerSignal sg{};
        for (int d = 0; d < ps.world; ++d) sg.flags[d] = reinterpret_cast<unsigned int *>(ps.base[d]);
        sg.rank = ps.rank; sg.world = ps.world; sg.epoch = epoch;
        sg.err = e->peer_err.p;
        sg.timeout_ns = 10ull * 1000ull * 1000ull * 1000ull;
        k_peer_signal_wait<<<1, 32, 0, e->stream>>>(sg);
        CK(cudaGetLastError());
        ++launches;
    }
    e->last_launches = launches + e->extra_launches;
    // status blocks back in the same breath; the synchronisation also keeps the pinned block ours until the next call
    std::vector<DevState> hst(n_rows);
    CK(cudaMemcpyAsync(hst.data(), st_dev, sizeof(DevState) * n_rows, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (e->timing) {
        e->t_k1 = e->t_k2 = e->t_k3 = 0;
        e->t_layer_k1.assign(n_layers, 0.f);
        e->t_layer_k2.assign(n_layers, 0.f);
        for (int bi = 0; bi < n_batches; ++bi) {
            const int b0 = (int)(bi * slots), b1 = (int)std::min<int64_t>(n_layers, b0 + slots);
            float a = 0, b = 0;
            CK(cudaEventElapsedTime(&a, e->ev[3 * bi], e->ev[3 * bi + 1]));
            CK(cudaEventElapsedTime(&b, e->ev[3 * bi + 1], e->ev[3 * bi + 2]));
            e->t_k1 += a;
            e->t_k2 += b;
            // per-layer figures are exact with one layer per batch (prb_set_option PRB_OPT_BATCH_LAYERS 0), else
            // the batch time spread evenly; reported in the caller's layer order
            for (int k = b0; k < b1; ++k) {
                const int l = pipe ? 0 : (int)(jobs[k].st_dev - st_dev);
                e->t_layer_k1[l] = a / (b1 - b0);
                e->t_layer_k2[l] = b / (b1 - b0);
            }
        }
        CK(cudaEventElapsedTime(&e->t_k3, e->ev[3 * n_batches], e->ev[3 * n_batches + 1]));
    }
    e->last.valid = false;
    if (ps.connected) {
        unsigned int perr = 0;
        CK(cudaMemcpy(&perr, e->peer_err.p, sizeof perr, cudaMemcpyDeviceToHost));
        if (perr) {
            CK(cudaMemset(e->peer_err.p, 0, sizeof perr));
            return fail(PRB_ERR_PEER, "peer gather timed out: a rank did not finish the step (ranks must call "
                                      "prb_atmosphere the same number of times)");
        }
    }
    return report_flags(hst.data(), n_rows);
}

extern "C" int prb_atmosphere(prb_engine *e, int32_t n_layers, int32_t n_groups, const double *depth_cm,
                              const double *t_layer, const double *p_layer, const double *conc, const double *molmass,
                              const double *q_t, const double *q_296, const int64_t *window_len, double t_surface,
                              double range_max) {
    return atmosphere_impl(e, n_layers, n_groups, depth_cm, t_layer, p_layer, conc, molmass, q_t, q_296, window_len,
                           t_surface, range_max, nullptr);
}

extern "C" int prb_atmosphere_result_dev(prb_engine *e, void **radiance_dev, void **transmittance_dev) {
    if (!e || !e->atm_layers) return fail(PRB_ERR_STATE, "prb_atmosphere_result_dev: run prb_atmosphere first");
    if (radiance_dev) *radiance_dev = e->res_rad;
    if (transmittance_dev) *transmittance_dev = e->res_trans;
    return PRB_OK;
}

extern "C" int prb_atmosphere_kmatrix_dev(prb_engine *e, void **kmat_dev, int64_t *ld) {
    if (!e || !e->atm_layers) return fail(PRB_ERR_STATE, "prb_atmosphere_kmatrix_dev: run prb_atmosphere first");
    if (kmat_dev) *kmat_dev = e->kmat.p;
    if (ld) *ld = e->kmat_ld;
    return PRB_OK;
}

extern "C" int prb_atmosphere_read(prb_engine *e, double *radiance_host, double *transmittance_host) {
    if (!e || !e->atm_layers) return fail(PRB_ERR_STATE, "prb_atmosphere_read: run prb_atmosphere first");
    CK(cudaSetDevice(e->device));
    const int64_t nc = chunk_len(e);
    // both spectra cross PCIe into one pinned staging block (grown on demand, kept), then widen to the caller's doubles
    if ((size_t)nc * 2 > e->read_stage_cap) {
        if (e->read_stage) cudaFreeHost(e->read_stage);
        e->read_stage = nullptr;
        e->read_stage_cap = 0;
        CK(cudaMallocHost((void **)&e->read_stage, sizeof(float) * std::max<size_t>((size_t)nc * 2, 1)));
        e->read_stage_cap = (size_t)nc * 2;
    }
    const float *src[2] = {e->res_rad, e->res_trans};
    double *dst[2] = {radiance_host, transmittance_host};
    for (int k = 0; k < 2; ++k)
        if (dst[k] && nc) CK(cudaMemcpyAsync(e->read_stage + (size_t)k * nc, src[k], sizeof(float) * nc, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    for (int k = 0; k < 2; ++k) {
        if (!dst[k]) continue;
        const float *t = e->read_stage + (size_t)k * nc;
        for (int64_t i = 0; i < nc; ++i) dst[k][i] = (double)t[i];
    }
    return PRB_OK;
}

extern "C" int prb_atmosphere_read_f32(prb_engine *e, float *radiance_host, float *transmittance_host) {
    if (!e || !e->atm_layers) return fail(PRB_ERR_STATE, "prb_atmosphere_read_f32: run prb_atmosphere first");
    CK(cudaSetDevice(e->device));
    const int64_t nc = chunk_len(e);
    if (radiance_host) CK(cudaMemcpyAsync(radiance_host, e->res_rad, sizeof(float) * nc, cudaMemcpyDeviceToHost, e->stream));
    if (transmittance_host)
        CK(cudaMemcpyAsync(transmittance_host, e->res_trans, sizeof(float) * nc, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return PRB_OK;
}

// One flux pass (k3_flux_tma) over the resident k matrix; its level sums (per CTA, or per segment for BAND) go to a.part.
template <int NMU, bool DOWN, bool BAND = false, bool BOUND = false, int SUN = K3F_NO_SUN>
static cudaError_t launch_flux(prb_engine *e, int grid, size_t smem, double dx, const K3FArgs &a) {
    const auto fn = k3_flux_tma<NMU, DOWN, BAND, BOUND, SUN>;
    cudaError_t ce = cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return ce;
    const double c2 = 100 * hPlanck * cLight / kBoltz;
    fn<<<grid, K3T_THREADS, smem, e->stream>>>(e->kmat.p, e->kmat_ld, e->atm_layers, e->flux_layers.p, chunk_len(e),
                                               e->i_begin, e->n_total, e->range_min, dx, e->atm_range_max,
                                               (float)(c2 / e->atm_t_surface), e->atm_nu_interp_min, a);
    return cudaGetLastError();
}

// SUN: the upward pass's solar variant (K3F_NO_SUN, K3F_SUN or K3F_SUN_SPECULAR); the downward pass carries the beam
// whenever there is one.
template <int NMU, bool BAND = false, bool BOUND = false, int SUN = K3F_NO_SUN>
static cudaError_t launch_flux_pair(prb_engine *e, int grid, size_t smem, double dx, const K3FArgs &up, const K3FArgs &down) {
    if constexpr (BOUND) {                             // the upward pass reflects the downward pass's surface rows
        constexpr int SUN_DOWN = SUN == K3F_NO_SUN ? K3F_NO_SUN : K3F_SUN;
        cudaError_t ce = launch_flux<NMU, true, BAND, true, SUN_DOWN>(e, grid, smem, dx, down);
        return ce != cudaSuccess ? ce : launch_flux<NMU, false, BAND, true, SUN>(e, grid, smem, dx, up);
    }
    cudaError_t ce = launch_flux<NMU, false, BAND>(e, grid, smem, dx, up);
    return ce != cudaSuccess ? ce : launch_flux<NMU, true, BAND>(e, grid, smem, dx, down);
}

template <bool BAND, bool BOUND, int SUN = K3F_NO_SUN>
static cudaError_t launch_flux_nodes(prb_engine *e, int n_mu, int grid, size_t smem, double dx, const K3FArgs &up,
                                     const K3FArgs &down) {
    switch (n_mu) {
        case 1: return launch_flux_pair<1, BAND, BOUND, SUN>(e, grid, smem, dx, up, down);
        case 2: return launch_flux_pair<2, BAND, BOUND, SUN>(e, grid, smem, dx, up, down);
        case 3: return launch_flux_pair<3, BAND, BOUND, SUN>(e, grid, smem, dx, up, down);
        default: return launch_flux_pair<4, BAND, BOUND, SUN>(e, grid, smem, dx, up, down);
    }
}

// A black surface, nothing from the top and no Sun: the plain passes.  A Sun takes the boundary passes.
static bool flux_bounded(const prb_engine *e) { return !e->bnd_tab.empty() || e->bnd_t_top > 0 || !e->sun_tab.empty(); }

template <bool BAND>
static cudaError_t launch_flux_passes(prb_engine *e, int n_mu, int grid, size_t smem, double dx, const K3FArgs &up,
                                      const K3FArgs &down) {
    if (!e->sun_tab.empty())
        return e->bnd_reflection == PRB_REFLECT_SPECULAR
                   ? launch_flux_nodes<BAND, true, K3F_SUN_SPECULAR>(e, n_mu, grid, smem, dx, up, down)
                   : launch_flux_nodes<BAND, true, K3F_SUN>(e, n_mu, grid, smem, dx, up, down);
    return flux_bounded(e) ? launch_flux_nodes<BAND, true>(e, n_mu, grid, smem, dx, up, down)
                           : launch_flux_nodes<BAND, false>(e, n_mu, grid, smem, dx, up, down);
}

// The radiance rows of the flux calls: up [0, 4), down [4, 8) and, with a Sun, the beam's row (8): S(nu) at the top,
// which the downward pass replaces with the beam at the surface.
static cudaError_t flux_rows_ensure(prb_engine *e) {
    return e->flux_rows.ensure((size_t)(e->sun_tab.empty() ? 8 : 9) * e->kmat_ld);
}

// With boundaries set: the emissivity on the chunk (k3_flux_emissivity, every call: the table is tiny), the downward
// pass's surface rows whether or not the caller reads them, and the boundary fields of both passes' arguments.
static cudaError_t flux_boundaries_prepare(prb_engine *e, double dx, K3FArgs &up, K3FArgs &down) {
    if (!flux_bounded(e)) return cudaSuccess;
    const int64_t nc = chunk_len(e);
    const std::vector<double> black{0.0, 1.0};        // no table: eps = 1 everywhere
    const std::vector<double> &tab = e->bnd_tab.empty() ? black : e->bnd_tab;
    const int64_t n_tab = (int64_t)tab.size() / 2;
    cudaError_t ce;
    if ((ce = flux_rows_ensure(e)) != cudaSuccess) return ce;
    if ((ce = e->flux_eps.ensure((size_t)e->kmat_ld)) != cudaSuccess) return ce;
    if ((ce = e->bnd_tab_dev.ensure(tab.size())) != cudaSuccess) return ce;
    ce = cudaMemcpyAsync(e->bnd_tab_dev.p, tab.data(), sizeof(double) * tab.size(), cudaMemcpyHostToDevice, e->stream);
    if (ce != cudaSuccess) return ce;
    const unsigned blocks = (unsigned)std::min<int64_t>((nc + 255) / 256, 8 * (int64_t)e->prop.multiProcessorCount);
    k3_flux_emissivity<<<blocks, 256, 0, e->stream>>>(nc, e->i_begin, e->n_total, e->range_min, dx, e->atm_range_max,
                                                      e->bnd_tab_dev.p, n_tab, e->flux_eps.p);
    if ((ce = cudaGetLastError()) != cudaSuccess) return ce;
    down.rows = e->flux_rows.p + (size_t)4 * e->kmat_ld;
    down.ld_rows = up.ld_rows = e->kmat_ld;
    down.c2_over_ttop = e->bnd_t_top > 0 ? (float)(100 * hPlanck * cLight / kBoltz / e->bnd_t_top) : 0.f;
    up.eps = e->flux_eps.p;
    up.surf_down = down.rows;
    up.specular = e->bnd_reflection == PRB_REFLECT_SPECULAR;
    if (e->sun_tab.empty()) return cudaSuccess;
    // the Sun: S on the chunk in the beam's row (k3_flux_solar, every call), and the beam's per-layer factors
    const int L = e->atm_layers;
    const int64_t n_sun = (int64_t)e->sun_tab.size() / 2;
    std::vector<float> nd(L);
    for (int l = 0; l < L; ++l) nd[l] = (float)(-e->atm_depth[l] * 1.4426950408889634 / e->sun_mu);
    if ((ce = e->sun_tab_dev.ensure(e->sun_tab.size())) != cudaSuccess) return ce;
    if ((ce = e->sun_nd.ensure((size_t)L)) != cudaSuccess) return ce;
    ce = cudaMemcpyAsync(e->sun_tab_dev.p, e->sun_tab.data(), sizeof(double) * e->sun_tab.size(), cudaMemcpyHostToDevice,
                         e->stream);
    if (ce != cudaSuccess) return ce;
    ce = cudaMemcpyAsync(e->sun_nd.p, nd.data(), sizeof(float) * L, cudaMemcpyHostToDevice, e->stream);
    if (ce != cudaSuccess) return ce;
    float *sun_row = e->flux_rows.p + (size_t)8 * e->kmat_ld;
    k3_flux_solar<<<blocks, 256, 0, e->stream>>>(nc, e->i_begin, e->n_total, e->range_min, dx, e->atm_range_max,
                                                 e->sun_tab_dev.p, n_sun, sun_row);
    if ((ce = cudaGetLastError()) != cudaSuccess) return ce;
    for (K3FArgs *a : {&up, &down}) {
        a->sun_nd = e->sun_nd.p;
        a->sun_w = (float)(e->sun_mu / (2 * 3.141592653589793));
    }
    up.sun_mu_over_pi = (float)(e->sun_mu / 3.141592653589793);
    return cudaSuccess;
}

// The checks shared by the flux calls: a column on the device, a quadrature of 1 to 4 nodes with mu in (0, 1] and finite
// weights > 0, and few enough layers for k3_flux_tma's per-level accumulators.
static int flux_check(prb_engine *e, const char *fn, int32_t n_mu, const double *mu, const double *weight) {
    if (!e || !e->atm_layers) return fail(PRB_ERR_STATE, std::string(fn) + ": run prb_atmosphere first");
    if (n_mu < 1 || n_mu > 4 || !mu || !weight) return fail(PRB_ERR_ARG, std::string(fn) + ": need 1 <= n_mu <= 4, mu and weight");
    for (int i = 0; i < n_mu; ++i)
        if (!(mu[i] > 0 && mu[i] <= 1) || !(weight[i] > 0 && std::isfinite(weight[i])))
            return fail(PRB_ERR_ARG, std::string(fn) + ": every mu must lie in (0, 1] and every weight be finite and > 0");
    if (k3f_smem_bytes(e->atm_layers) > (size_t)e->prop.sharedMemPerBlockOptin)
        return fail(PRB_ERR_RANGE, std::string(fn) + ": too many layers for the per-level accumulators in shared memory");
    return PRB_OK;
}

// Per layer: c2 / T_l and -depth_l log2(e) / mu_i, rounded as the fold rounds them (mu = 1 gives its very constants),
// uploaded to e->flux_layers; and w_i mu_i into both passes' arguments.
static cudaError_t flux_layers_upload(prb_engine *e, int32_t n_mu, const double *mu, const double *weight,
                                      std::vector<FluxLayer> &hl, K3FArgs &up, K3FArgs &down) {
    const int L = e->atm_layers;
    const double c2 = 100 * hPlanck * cLight / kBoltz;
    hl.resize(L);
    for (int l = 0; l < L; ++l) {
        hl[l].c2_over_t = (float)(c2 / e->atm_t[l]);
        for (int i = 0; i < 4; ++i) hl[l].nd[i] = i < n_mu ? (float)(-e->atm_depth[l] * 1.4426950408889634 / mu[i]) : 0.f;
    }
    for (int i = 0; i < n_mu; ++i) up.wmu[i] = down.wmu[i] = (float)(weight[i] * mu[i]);
    cudaError_t ce = e->flux_layers.ensure(L);
    if (ce != cudaSuccess) return ce;
    return cudaMemcpyAsync(e->flux_layers.p, hl.data(), sizeof(FluxLayer) * L, cudaMemcpyHostToDevice, e->stream);
}

static double flux_dx(const prb_engine *e) {
    return e->n_total > 1 ? (e->atm_range_max - e->range_min) / (double)(e->n_total - 1) : 0.0;
}

extern "C" int prb_atmosphere_fluxes(prb_engine *e, int32_t n_mu, const double *mu, const double *weight, double *flux_up,
                                     double *flux_down, float *rad_up_top, float *rad_down_surface) {
    if (int rc = flux_check(e, "prb_atmosphere_fluxes", n_mu, mu, weight)) return rc;
    CK(cudaSetDevice(e->device));
    const int L = e->atm_layers, n_levels = L + 1;
    const int64_t nc = chunk_len(e);
    const size_t smem = k3f_smem_bytes(L);
    if (nc == 0) {                                              // an empty chunk contributes nothing
        if (flux_up) std::fill(flux_up, flux_up + n_levels, 0.0);
        if (flux_down) std::fill(flux_down, flux_down + n_levels, 0.0);
        return PRB_OK;
    }
    std::vector<FluxLayer> hl;
    K3FArgs up{}, down{};
    CK(flux_layers_upload(e, n_mu, mu, weight, hl, up, down));
    const int64_t n_strips = (nc + K3T_STRIP - 1) / K3T_STRIP;
    const int grid = (int)std::min<int64_t>(n_strips, k3f_minb(n_mu) * (int64_t)e->prop.multiProcessorCount);
    const bool rows = rad_up_top || rad_down_surface;
    CK(e->flux_part.ensure((size_t)2 * grid * n_levels));
    CK(e->flux_out.ensure((size_t)2 * n_levels));
    if (rows) CK(flux_rows_ensure(e));
    up.ld_rows = down.ld_rows = e->kmat_ld;
    up.rows = rows ? e->flux_rows.p : nullptr;
    down.rows = rows ? e->flux_rows.p + (size_t)4 * e->kmat_ld : nullptr;
    up.part = e->flux_part.p;
    down.part = e->flux_part.p + (size_t)grid * n_levels;
    CK(flux_boundaries_prepare(e, flux_dx(e), up, down));
    const cudaError_t ce = launch_flux_passes<false>(e, n_mu, grid, smem, flux_dx(e), up, down);
    if (ce != cudaSuccess) return fail(PRB_ERR_CUDA, std::string("k3_flux_tma launch failed: ") + cudaGetErrorString(ce));
    // F[j] = 2 pi sum_i w_i mu_i sum_nu I_i(nu, j) res  (integrateSpectrum's res and NaN rule, pyradClasses.py:26-29)
    const double scale = 2 * 3.141592653589793 * e->res;
    const unsigned sum_blocks = (unsigned)((n_levels + 255) / 256);
    k3_flux_sum<<<sum_blocks, 256, 0, e->stream>>>(up.part, grid, n_levels, scale, e->flux_out.p);
    k3_flux_sum<<<sum_blocks, 256, 0, e->stream>>>(down.part, grid, n_levels, scale, e->flux_out.p + n_levels);
    CK(cudaGetLastError());
    if (flux_up) CK(cudaMemcpyAsync(flux_up, e->flux_out.p, sizeof(double) * n_levels, cudaMemcpyDeviceToHost, e->stream));
    if (flux_down)
        CK(cudaMemcpyAsync(flux_down, e->flux_out.p + n_levels, sizeof(double) * n_levels, cudaMemcpyDeviceToHost, e->stream));
    for (int i = 0; i < n_mu; ++i) {
        if (rad_up_top)
            CK(cudaMemcpyAsync(rad_up_top + (size_t)i * nc, up.rows + (size_t)i * e->kmat_ld, sizeof(float) * nc,
                               cudaMemcpyDeviceToHost, e->stream));
        if (rad_down_surface)
            CK(cudaMemcpyAsync(rad_down_surface + (size_t)i * nc, down.rows + (size_t)i * e->kmat_ld, sizeof(float) * nc,
                               cudaMemcpyDeviceToHost, e->stream));
    }
    CK(cudaStreamSynchronize(e->stream));
    return PRB_OK;
}

// The first grid point i in [0, n] with axis_value(i) >= v (n if none): the axis is non-decreasing.
static int64_t first_point_at_or_above(double v, int64_t n, double x0, double dx, double x_last) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = lo + (hi - lo) / 2;
        if (axis_value(mid, n, x0, dx, x_last) >= v) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}

extern "C" int prb_atmosphere_band_fluxes(prb_engine *e, int32_t n_mu, const double *mu, const double *weight,
                                          int32_t n_bands, const double *edges, double *band_up, double *band_down) {
    if (int rc = flux_check(e, "prb_atmosphere_band_fluxes", n_mu, mu, weight)) return rc;
    if (n_bands < 1 || !edges) return fail(PRB_ERR_ARG, "prb_atmosphere_band_fluxes: need n_bands >= 1 and n_bands + 1 edges");
    for (int b = 0; b <= n_bands; ++b)
        if (!std::isfinite(edges[b]) || (b > 0 && !(edges[b] > edges[b - 1])))
            return fail(PRB_ERR_ARG, "prb_atmosphere_band_fluxes: the edges must be finite and strictly ascending");
    CK(cudaSetDevice(e->device));
    const int L = e->atm_layers, n_levels = L + 1;
    const int64_t nc = chunk_len(e);
    const size_t per_dir = (size_t)n_bands * n_levels;
    auto zeros = [&]() {
        if (band_up) std::fill(band_up, band_up + per_dir, 0.0);
        if (band_down) std::fill(band_down, band_down + per_dir, 0.0);
        return PRB_OK;
    };
    if (nc == 0) return zeros();                                // an empty chunk contributes nothing
    constexpr int SPAN = 128;                                   // points per warp
    const int64_t n_strips = (nc + K3T_STRIP - 1) / K3T_STRIP, n_spans = n_strips * K3F_WARPS;
    if (n_spans + n_bands + 1 > INT32_MAX) return fail(PRB_ERR_RANGE, "prb_atmosphere_band_fluxes: chunk too long");
    // Band b holds the points with edges[b] <= x_i < edges[b+1], x the Planck axis of the fold: the chunk-local points
    // [p[b], p[b+1]), each p the first point at or above its edge by the device's own formula (exact at grid values).
    const double dx = flux_dx(e);
    std::vector<int64_t> p(n_bands + 1);
    for (int b = 0; b <= n_bands; ++b)
        p[b] = std::clamp<int64_t>(first_point_at_or_above(edges[b], e->n_total, e->range_min, dx, e->atm_range_max) -
                                   e->i_begin, 0, nc);
    // Segments (span x band) in position order; a band's segments are consecutive: band_seg[b] .. band_seg[b+1].
    std::vector<K3FSpan> spans(n_spans, K3FSpan{0, 0});
    std::vector<uint32_t> seg_range;
    std::vector<int32_t> band_seg(n_bands + 1);
    for (int b = 0; b < n_bands; ++b) {
        band_seg[b] = (int32_t)seg_range.size();
        if (p[b] >= p[b + 1]) continue;                         // a band with no points: no segments, zeros
        for (int64_t s = p[b] / SPAN; s <= (p[b + 1] - 1) / SPAN; ++s) {
            const int64_t s0 = s * SPAN, s1 = std::min(s0 + SPAN, nc);
            const uint32_t lo = (uint32_t)(std::max(p[b], s0) - s0), hi = (uint32_t)(std::min(p[b + 1], s1) - s0);
            if (spans[s].nseg == 0) spans[s].seg0 = (int32_t)seg_range.size();
            spans[s].nseg++;
            seg_range.push_back(lo | hi << 16);
        }
    }
    const int64_t n_seg = (int64_t)seg_range.size();
    band_seg[n_bands] = (int32_t)n_seg;
    for (int64_t s = 0; s < n_spans; ++s)                       // one band over all of the span's points: the plain sum
        if (spans[s].nseg == 1 && seg_range[spans[s].seg0] == (uint32_t)(std::min<int64_t>(SPAN, nc - s * SPAN) << 16))
            spans[s].nseg = -1;
    // the strips that meet a band, and the bands by the size of their sum (k3_flux_band_sum)
    std::vector<int32_t> strips, small, big;
    for (int64_t t = 0; t < n_strips; ++t)
        for (int w = 0; w < K3F_WARPS; ++w)
            if (spans[t * K3F_WARPS + w].nseg != 0) { strips.push_back((int32_t)t); break; }
    if (strips.empty()) return zeros();                         // no band meets the chunk
    for (int b = 0; b < n_bands; ++b) (band_seg[b + 1] - band_seg[b] > K3F_BAND_WARP_MAX ? big : small).push_back(b);
    // one upload: spans | seg_range | band_seg | strips | small | big
    std::vector<int32_t> tab(2 * n_spans + n_seg);
    std::memcpy(tab.data(), spans.data(), sizeof(K3FSpan) * n_spans);
    std::memcpy(tab.data() + 2 * n_spans, seg_range.data(), sizeof(uint32_t) * n_seg);
    const size_t o_band = tab.size(), o_strips = o_band + band_seg.size(), o_small = o_strips + strips.size(),
                 o_big = o_small + small.size();
    for (const auto *v : {&band_seg, &strips, &small, &big}) tab.insert(tab.end(), v->begin(), v->end());
    std::vector<FluxLayer> hl;
    K3FArgs up{}, down{};
    CK(flux_layers_upload(e, n_mu, mu, weight, hl, up, down));
    CK(e->band_tab.ensure(tab.size()));
    CK(cudaMemcpyAsync(e->band_tab.p, tab.data(), sizeof(int32_t) * tab.size(), cudaMemcpyHostToDevice, e->stream));
    CK(e->band_part.ensure((size_t)2 * n_levels * n_seg));
    CK(e->band_out.ensure(2 * per_dir));
    const int32_t *d_tab = e->band_tab.p;
    for (K3FArgs *a : {&up, &down}) {
        a->strips = d_tab + o_strips;
        a->n_list = (int64_t)strips.size();
        a->spans = reinterpret_cast<const K3FSpan *>(d_tab);
        a->seg_range = reinterpret_cast<const uint32_t *>(d_tab + 2 * n_spans);
        a->ld_part = n_seg;
    }
    up.part = e->band_part.p;
    down.part = e->band_part.p + (size_t)n_levels * n_seg;
    CK(flux_boundaries_prepare(e, dx, up, down));
    const int grid = (int)std::min<int64_t>((int64_t)strips.size(), k3f_minb(n_mu) * (int64_t)e->prop.multiProcessorCount);
    const cudaError_t ce = launch_flux_passes<true>(e, n_mu, grid, sizeof(K3FSmem), dx, up, down);
    if (ce != cudaSuccess) return fail(PRB_ERR_CUDA, std::string("k3_flux_tma launch failed: ") + cudaGetErrorString(ce));
    // F_b[j] = 2 pi sum_i w_i mu_i sum_{nu in band b} I_i(nu, j) res
    const double scale = 2 * 3.141592653589793 * e->res;
    if (!small.empty()) {
        const int64_t items = 2 * (int64_t)small.size() * n_levels;
        k3_flux_band_sum<32><<<(unsigned)((items + 7) / 8), 256, 0, e->stream>>>(
            e->band_part.p, n_seg, n_levels, d_tab + o_small, (int)small.size(), d_tab + o_band, n_bands, scale, e->band_out.p);
    }
    if (!big.empty())
        k3_flux_band_sum<256><<<(unsigned)(2 * big.size() * n_levels), 256, 0, e->stream>>>(
            e->band_part.p, n_seg, n_levels, d_tab + o_big, (int)big.size(), d_tab + o_band, n_bands, scale, e->band_out.p);
    CK(cudaGetLastError());
    if (band_up) CK(cudaMemcpyAsync(band_up, e->band_out.p, sizeof(double) * per_dir, cudaMemcpyDeviceToHost, e->stream));
    if (band_down)
        CK(cudaMemcpyAsync(band_down, e->band_out.p + per_dir, sizeof(double) * per_dir, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return PRB_OK;
}

extern "C" int prb_set_flux_boundaries(prb_engine *e, int64_t n_table, const double *table_nu,
                                       const double *table_emissivity, int32_t reflection, double t_top) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n_table < 0 || (n_table > 0 && (!table_nu || !table_emissivity)))
        return fail(PRB_ERR_ARG, "prb_set_flux_boundaries: need n_table >= 0 and both tables when n_table > 0");
    for (int64_t i = 0; i < n_table; ++i) {
        if (!std::isfinite(table_nu[i]) || (i > 0 && !(table_nu[i] > table_nu[i - 1])))
            return fail(PRB_ERR_ARG, "prb_set_flux_boundaries: table_nu must be finite and strictly ascending");
        if (!(table_emissivity[i] >= 0 && table_emissivity[i] <= 1))
            return fail(PRB_ERR_ARG, "prb_set_flux_boundaries: every emissivity must lie in [0, 1]");
    }
    if (reflection != PRB_REFLECT_LAMBERTIAN && reflection != PRB_REFLECT_SPECULAR)
        return fail(PRB_ERR_ARG, "prb_set_flux_boundaries: reflection must be PRB_REFLECT_LAMBERTIAN or PRB_REFLECT_SPECULAR");
    if (!(std::isfinite(t_top) && t_top >= 0))
        return fail(PRB_ERR_ARG, "prb_set_flux_boundaries: t_top must be finite and >= 0");
    e->bnd_tab.assign(table_nu, table_nu + n_table);
    e->bnd_tab.insert(e->bnd_tab.end(), table_emissivity, table_emissivity + n_table);
    e->bnd_reflection = reflection;
    e->bnd_t_top = t_top;
    return PRB_OK;
}

extern "C" int prb_set_solar_source(prb_engine *e, int64_t n_table, const double *table_nu,
                                    const double *table_irradiance, double mu_sun) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n_table == 0) {
        e->sun_tab.clear();
        return PRB_OK;
    }
    if (n_table < 2 || !table_nu || !table_irradiance)
        return fail(PRB_ERR_ARG, "prb_set_solar_source: need n_table = 0, or n_table >= 2 and both tables");
    for (int64_t i = 0; i < n_table; ++i) {
        if (!std::isfinite(table_nu[i]) || (i > 0 && !(table_nu[i] > table_nu[i - 1])))
            return fail(PRB_ERR_ARG, "prb_set_solar_source: table_nu must be finite and strictly ascending");
        if (!(std::isfinite(table_irradiance[i]) && table_irradiance[i] >= 0))
            return fail(PRB_ERR_ARG, "prb_set_solar_source: every irradiance must be finite and >= 0");
    }
    if (!(mu_sun > 0 && mu_sun <= 1)) return fail(PRB_ERR_ARG, "prb_set_solar_source: mu_sun must lie in (0, 1]");
    e->sun_tab.assign(table_nu, table_nu + n_table);
    e->sun_tab.insert(e->sun_tab.end(), table_irradiance, table_irradiance + n_table);
    e->sun_mu = mu_sun;
    return PRB_OK;
}

extern "C" int prb_set_timing(prb_engine *e, int enabled) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    e->timing = enabled != 0;
    return PRB_OK;
}

extern "C" int prb_atmosphere_timing(prb_engine *e, float *k1_ms, float *k2_ms, float *k3_ms) {
    if (!e || !e->atm_layers || !e->timing) return fail(PRB_ERR_STATE, "prb_atmosphere_timing: enable timing and run prb_atmosphere first");
    if (k1_ms) *k1_ms = e->t_k1;
    if (k2_ms) *k2_ms = e->t_k2;
    if (k3_ms) *k3_ms = e->t_k3;
    return PRB_OK;
}

extern "C" int prb_atmosphere_layer_timing(prb_engine *e, int32_t n_layers, float *k1_ms, float *k2_ms) {
    if (!e || !e->atm_layers || !e->timing || (int)e->t_layer_k1.size() != n_layers)
        return fail(PRB_ERR_STATE, "prb_atmosphere_layer_timing: enable timing, run prb_atmosphere, pass its layer count");
    for (int l = 0; l < n_layers; ++l) {
        if (k1_ms) k1_ms[l] = e->t_layer_k1[l];
        if (k2_ms) k2_ms[l] = e->t_layer_k2[l];
    }
    return PRB_OK;
}

extern "C" int prb_set_narrow_threshold(prb_engine *e, int64_t wm_below) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    e->narrow_wm = wm_below < 0 ? 100 : wm_below;
    e->last.valid = false;                                      // record layout may change: redo the prepass
    return PRB_OK;
}

extern "C" int prb_set_option(prb_engine *e, int option, int64_t value) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    switch (option) {
        case PRB_OPT_BATCH_LAYERS: e->batch_layers = value != 0; return PRB_OK;
        case PRB_OPT_FUSE_SINGLE_LAYER: e->fuse_single = value != 0; return PRB_OK;
        case PRB_OPT_POINT_KERNEL: e->point_kernel = value != 0; e->last.valid = false; return PRB_OK;
        case PRB_OPT_FOLD_TMA: e->k3_tma = value != 0; return PRB_OK;
        case PRB_OPT_SPLIT_TILES: e->split_tiles = value != 0; return PRB_OK;
        case PRB_OPT_RECORD_BUDGET_MB: e->rec_budget_mb = value < 0 ? 0 : value; return PRB_OK;
        default: return fail(PRB_ERR_ARG, "prb_set_option: unknown option");
    }
}

extern "C" int prb_atmosphere_launches(prb_engine *e) { return e ? e->last_launches : 0; }

// ------------------------------------------------------------------------------------ peer gather (multi-GPU)
// One process per GPU on one NVLink / NVSwitch node.  Each rank allocates a gather buffer, exports it as a CUDA
// IPC handle; the host side exchanges the 64-byte handles by whatever transport it has (torch.distributed in
// pyrad_b200/distributed.py, MPI, a file) and hands all of them back.  From then on prb_atmosphere stores this
// rank's finished spectra straight into every rank's buffer from inside its last kernel and ends with a cross-GPU
// flag barrier, so the all-gather of the spectra is part of the compute step (no separate collective).
extern "C" int prb_peer_alloc(prb_engine *e, int rank, int world, int64_t max_chunk_points, void *handle_out) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (world < 1 || world > K2_MAX_PEERS || rank < 0 || rank >= world)
        return fail(PRB_ERR_ARG, "prb_peer_alloc: world must be 1..8 and 0 <= rank < world");
    if (max_chunk_points < 1 || !handle_out) return fail(PRB_ERR_ARG, "prb_peer_alloc: bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == PRB_PEER_HANDLE_BYTES, "handle size");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    peer_release(e);
    PeerState &ps = e->peer;
    ps.rank = rank; ps.world = world;
    ps.ld = (max_chunk_points + 63) & ~int64_t(63);
    ps.bytes = PEER_HEADER + (size_t)2 * 2 * world * (size_t)ps.ld * sizeof(float);
    CK(cudaMalloc((void **)&ps.local, ps.bytes));
    CK(cudaMemset(ps.local, 0, ps.bytes));
    CK(e->peer_err.ensure(1));
    CK(cudaMemset(e->peer_err.p, 0, sizeof(unsigned int)));
    cudaIpcMemHandle_t hd;
    CK(cudaIpcGetMemHandle(&hd, ps.local));
    memcpy(handle_out, &hd, sizeof hd);
    return PRB_OK;
}

extern "C" int prb_peer_connect(prb_engine *e, const void *handles) {
    if (!e || !handles) return fail(PRB_ERR_ARG, "prb_peer_connect: bad arguments");
    PeerState &ps = e->peer;
    if (!ps.local) return fail(PRB_ERR_STATE, "prb_peer_connect: call prb_peer_alloc first");
    if (ps.connected) return fail(PRB_ERR_STATE, "prb_peer_connect: already connected");
    CK(cudaSetDevice(e->device));
    for (int r = 0; r < ps.world; ++r) {
        if (r == ps.rank) { ps.base[r] = ps.local; continue; }
        cudaIpcMemHandle_t hd;
        memcpy(&hd, (const unsigned char *)handles + (size_t)r * sizeof hd, sizeof hd);
        void *ptr = nullptr;
        cudaError_t ce = cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess);
        if (ce != cudaSuccess) {
            for (int q = 0; q < r; ++q) if (q != ps.rank && ps.base[q]) { cudaIpcCloseMemHandle(ps.base[q]); ps.base[q] = nullptr; }
            return fail(PRB_ERR_PEER, std::string("prb_peer_connect: cudaIpcOpenMemHandle failed for rank ") +
                                          std::to_string(r) + ": " + cudaGetErrorString(ce));
        }
        ps.base[r] = (unsigned char *)ptr;
    }
    ps.connected = true;
    ps.epoch = 0;
    return PRB_OK;
}

extern "C" int prb_peer_disconnect(prb_engine *e) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    peer_release(e);
    e->res_rad = e->res_trans = nullptr;
    e->atm_layers = 0;
    return PRB_OK;
}

extern "C" int prb_peer_gathered_dev(prb_engine *e, void **radiance_dev, void **transmittance_dev, int64_t *ld) {
    if (!e || !e->peer.connected || !e->peer.epoch)
        return fail(PRB_ERR_STATE, "prb_peer_gathered_dev: connect the peers and run prb_atmosphere first");
    const int par = e->peer.epoch & 1;
    if (radiance_dev) *radiance_dev = peer_slot(e, e->peer.rank, par, 0, 0);
    if (transmittance_dev) *transmittance_dev = peer_slot(e, e->peer.rank, par, 1, 0);
    if (ld) *ld = e->peer.ld;
    return PRB_OK;
}

// ------------------------------------------------------------------------------------ K4: survey, integrals, derived
extern "C" int prb_line_survey(prb_engine *e, int64_t n_out, double *out_host) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (!e->grid_set) return fail(PRB_ERR_STATE, "prb_line_survey: upload lines and set the grid first");
    if (n_out < 0 || (n_out > 0 && !out_host)) return fail(PRB_ERR_ARG, "prb_line_survey: bad arguments");
    if (n_out == 0) return PRB_OK;
    CK(cudaSetDevice(e->device));
    CK(e->scratch_b.ensure(n_out));
    CK(cudaMemsetAsync(e->scratch_b.p, 0, sizeof(double) * n_out, e->stream));
    if (e->n_lines > 0) {
        k4_line_survey<<<(unsigned)((e->n_lines + 255) / 256), 256, 0, e->stream>>>(e->idx.p, e->s296.p, e->n_lines, n_out,
                                                                                  e->scratch_b.p);
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(out_host, e->scratch_b.p, sizeof(double) * n_out, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return PRB_OK;
}

template <typename T>
static int device_sum(prb_engine *e, const T *x_dev, int64_t n, double scale, double *out_host) {
    const int64_t per_block = (int64_t)K4_BLOCK * K4_PER_THREAD;
    const int64_t nb = std::max<int64_t>(1, (n + per_block - 1) / per_block);
    CK(e->scratch_w.ensure(nb + 1));
    k4_sum_partial<T><<<(unsigned)nb, K4_BLOCK, 0, e->stream>>>(x_dev, n, e->scratch_w.p);
    CK(cudaGetLastError());
    k4_sum_final<<<1, K4_BLOCK, 0, e->stream>>>(e->scratch_w.p, nb, scale, e->scratch_w.p + nb);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out_host, e->scratch_w.p + nb, sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return PRB_OK;
}

extern "C" int prb_integrate_spectrum(prb_engine *e, int64_t n, const double *spectrum, double unit_angle, double res,
                                      double *value) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n < 0 || (n > 0 && !spectrum) || !value) return fail(PRB_ERR_ARG, "prb_integrate_spectrum: bad arguments");
    CK(cudaSetDevice(e->device));
    CK(e->scratch_a.ensure(std::max<int64_t>(n, 1)));
    if (n) CK(cudaMemcpyAsync(e->scratch_a.p, spectrum, sizeof(double) * n, cudaMemcpyHostToDevice, e->stream));
    // value = sum * unitAngle * res, left to right as the reference (pyradClasses.py:27-28)
    double sum = 0;
    int rc = device_sum<double>(e, e->scratch_a.p, n, 1.0, &sum);
    if (rc) return rc;
    *value = sum * unit_angle * res;
    return PRB_OK;
}

extern "C" int prb_atmosphere_integrate(prb_engine *e, double unit_angle, double res, double *radiance_integral,
                                        double *transmittance_sum) {
    if (!e || !e->atm_layers || !e->res_rad)
        return fail(PRB_ERR_STATE, "prb_atmosphere_integrate: run prb_atmosphere first");
    CK(cudaSetDevice(e->device));
    const int64_t nc = chunk_len(e);
    int rc;
    if (radiance_integral) {
        double s = 0;
        if ((rc = device_sum<float>(e, e->res_rad, nc, 1.0, &s))) return rc;
        *radiance_integral = s * unit_angle * res;
    }
    if (transmittance_sum) {
        if ((rc = device_sum<float>(e, e->res_trans, nc, 1.0, transmittance_sum))) return rc;
    }
    return PRB_OK;
}

extern "C" int prb_derived_spectra(prb_engine *e, int64_t n, const double *transmittance, double *emissivity,
                                   double *optical_depth, double *absorbance) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n < 0 || (n > 0 && !transmittance)) return fail(PRB_ERR_ARG, "prb_derived_spectra: bad arguments");
    if (n == 0) return PRB_OK;
    CK(cudaSetDevice(e->device));
    CK(e->scratch_a.ensure(n)); CK(e->scratch_b.ensure(n)); CK(e->scratch_c.ensure(n)); CK(e->scratch_d.ensure(n));
    CK(cudaMemcpyAsync(e->scratch_a.p, transmittance, sizeof(double) * n, cudaMemcpyHostToDevice, e->stream));
    k4_derived_f64<<<stream_grid(e, n), 256, 0, e->stream>>>(n, e->scratch_a.p, emissivity ? e->scratch_b.p : nullptr,
                                                            optical_depth ? e->scratch_c.p : nullptr,
                                                            absorbance ? e->scratch_d.p : nullptr);
    CK(cudaGetLastError());
    if (emissivity) CK(cudaMemcpyAsync(emissivity, e->scratch_b.p, sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    if (optical_depth) CK(cudaMemcpyAsync(optical_depth, e->scratch_c.p, sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    if (absorbance) CK(cudaMemcpyAsync(absorbance, e->scratch_d.p, sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return PRB_OK;
}

// ------------------------------------------------------------------------------------ K5: HITRAN CSV ingestion
extern "C" int prb_ingest_hitran_csv(prb_engine *e, const char *text, int64_t n_bytes, double wave_min, double wave_max,
                                     int64_t *n_lines_out) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n_bytes < 0 || (n_bytes > 0 && !text)) return fail(PRB_ERR_ARG, "prb_ingest_hitran_csv: bad arguments");
    if (n_bytes > (int64_t(1) << 36)) return fail(PRB_ERR_ARG, "prb_ingest_hitran_csv: more than 64 GiB of text; ingest in pieces");
    CK(cudaSetDevice(e->device));
    auto lap = [&](const char *) {};                             // (phase timing hook of the development builds)
    const int64_t n_pad = std::max<int64_t>((n_bytes + 15) & ~int64_t(15), 16);
    // scratch lives in the engine and only grows (device allocation is far slower than the parse itself)
    IngestScratch &g = e->ingest;
    DevBuf<char> &d_text = g.text;
    DevBuf<unsigned char> &d_nl = g.nl, &d_state = g.state, &d_tmp = g.tmp;
    DevBuf<int32_t> &d_keep = g.keep, &d_pos = g.pos;
    DevBuf<int64_t> &d_nlpos = g.nlpos;
    DevBuf<unsigned long long> &d_scal = g.scal;   // [0] newline count, [1] first bad row, [2] smax bits, [3] unsorted flag, [4] selected
    DevBuf<double> *t = g.cols;
    auto cleanup = [&]() {};
#define CKI(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); char b_[512]; \
        snprintf(b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
        return fail(PRB_ERR_CUDA, b_); } } while (0)
    CKI(d_text.ensure(n_pad));
    CKI(d_nl.ensure(n_pad));
    CKI(d_scal.ensure(8));
    CKI(cudaMemsetAsync(d_text.p + (n_pad - 16), 0, 16, e->stream));
    if (n_bytes) CKI(cudaMemcpyAsync(d_text.p, text, n_bytes, cudaMemcpyHostToDevice, e->stream));
    unsigned long long h_scal[8] = {0, ~0ull, 0, 0, 0, 0, 0, 0};
    CKI(cudaMemcpyAsync(d_scal.p, h_scal, sizeof h_scal, cudaMemcpyHostToDevice, e->stream));
    lap("alloc + H2D text");
    k5_mark_newlines<<<(unsigned)((n_pad / 16 + 255) / 256), 256, 0, e->stream>>>(d_text.p, n_bytes, d_nl.p, d_scal.p);
    CKI(cudaGetLastError());
    CKI(cudaMemcpyAsync(h_scal, d_scal.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream));
    CKI(cudaStreamSynchronize(e->stream));
    lap("mark newlines");
    const int64_t n_nl = (int64_t)h_scal[0];
    const int64_t n_rows = n_nl + ((n_bytes > 0 && text[n_bytes - 1] != '\n') ? 1 : 0);
    int64_t n_kept = 0;
    if (n_rows > 0) {
        // newline positions (CUB stream compaction of a counting sequence)
        CKI(d_nlpos.ensure(n_nl + 1));
        size_t tmp_bytes = 0;
        thrust::counting_iterator<int64_t> counting(0);
        long long *d_selected = reinterpret_cast<long long *>(d_scal.p + 4);
        CKI(cub::DeviceSelect::Flagged(nullptr, tmp_bytes, counting, d_nl.p, d_nlpos.p, d_selected, n_bytes, e->stream));
        CKI(d_tmp.ensure(tmp_bytes));
        CKI(cub::DeviceSelect::Flagged(d_tmp.p, tmp_bytes, counting, d_nl.p, d_nlpos.p, d_selected, n_bytes, e->stream));
        lap("newline positions (CUB)");
        for (int c = 0; c < 8; ++c) CKI(t[c].ensure(n_rows));
        CKI(d_state.ensure(n_rows));
        CKI(d_keep.ensure(n_rows));
        CKI(d_pos.ensure(n_rows + 1));
        IngestCols tc{t[0].p, t[1].p, t[2].p, t[3].p, t[4].p, t[5].p, t[6].p, t[7].p};
        k5_parse_rows<<<(unsigned)((n_rows + K5_ROWS - 1) / K5_ROWS), K5_ROWS, 0, e->stream>>>(d_text.p, n_bytes, d_nlpos.p, n_nl, n_rows, wave_min,
                                                                             wave_max, tc, d_state.p, d_scal.p + 1);
        CKI(cudaGetLastError());
        lap("alloc rows + parse");
        k5_resolve_duplicates<<<(unsigned)((n_rows + 255) / 256), 256, 0, e->stream>>>(t[0].p, d_state.p, n_rows, d_keep.p);
        CKI(cudaGetLastError());
        // exclusive scan of the keep flags -> output slots
        size_t tmp2 = 0;
        CKI(cub::DeviceScan::ExclusiveSum(nullptr, tmp2, d_keep.p, d_pos.p, n_rows, e->stream));
        CKI(d_tmp.ensure(tmp2));
        CKI(cub::DeviceScan::ExclusiveSum(d_tmp.p, tmp2, d_keep.p, d_pos.p, n_rows, e->stream));
        int32_t last_pos = 0, last_keep = 0;
        CKI(cudaMemcpyAsync(&last_pos, d_pos.p + (n_rows - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
        CKI(cudaMemcpyAsync(&last_keep, d_keep.p + (n_rows - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
        CKI(cudaMemcpyAsync(h_scal, d_scal.p, sizeof h_scal, cudaMemcpyDeviceToHost, e->stream));
        CKI(cudaStreamSynchronize(e->stream));
        if (h_scal[1] != ~0ull) {
            cleanup();
            return fail(PRB_ERR_PARSE, "prb_ingest_hitran_csv: row " + std::to_string(h_scal[1]) +
                                           " is not a HITRAN-online CSV row (10 comma-separated fields, plain decimal numbers)");
        }
        lap("duplicates + scan");
        n_kept = (int64_t)last_pos + last_keep;
        e->lines_set = false;
        int rc = alloc_line_storage(e, n_kept);
        if (rc) { cleanup(); return rc; }
        IngestCols dst{e->nu0.p, e->s296.p, e->einstein_a.p, e->elower.p, e->gair.p, e->gself.p, e->delta.p, e->nair.p};
        k5_scatter_kept<<<(unsigned)((n_rows + 255) / 256), 256, 0, e->stream>>>(tc, d_keep.p, d_pos.p, n_rows, dst);
        CKI(cudaGetLastError());
        if (n_kept > 0) {
            k5_finalize<<<(unsigned)((n_kept + 255) / 256), 256, 0, e->stream>>>(e->nu0.p, e->s296.p, n_kept, d_scal.p + 2,
                                                                               reinterpret_cast<unsigned int *>(d_scal.p + 3));
            CKI(cudaGetLastError());
        }
        CKI(cudaMemcpyAsync(h_scal, d_scal.p, sizeof h_scal, cudaMemcpyDeviceToHost, e->stream));
        CKI(cudaStreamSynchronize(e->stream));
        if ((h_scal[3] & 0xffffffffull) && n_kept > 1) {
            // out of order: stable radix sort of the kept rows by wavenumber, last row of every equal-wavenumber run wins,
            // columns gathered back into the engine's SoA (the parse buffers t[] serve as the source copy)
            IngestCols cur{e->nu0.p, e->s296.p, e->einstein_a.p, e->elower.p, e->gair.p, e->gself.p, e->delta.p, e->nair.p};
            const unsigned gk = (unsigned)((n_kept + 255) / 256);
            for (int c = 0; c < 8; ++c) {
                double *src8[8] = {cur.nu, cur.sw, cur.a, cur.elower, cur.gair, cur.gself, cur.delta, cur.nair};
                CKI(cudaMemcpyAsync(t[c].p, src8[c], sizeof(double) * n_kept, cudaMemcpyDeviceToDevice, e->stream));
            }
            DevBuf<double> keys_out;
            DevBuf<int32_t> perm_in, perm_out;
            CKI(keys_out.ensure(n_kept)); CKI(perm_in.ensure(n_kept)); CKI(perm_out.ensure(n_kept));
            k5_iota<<<gk, 256, 0, e->stream>>>(perm_in.p, n_kept);
            size_t tmp3 = 0;
            CKI(cub::DeviceRadixSort::SortPairs(nullptr, tmp3, t[0].p, keys_out.p, perm_in.p, perm_out.p, (int)n_kept, 0, 64, e->stream));
            CKI(d_tmp.ensure(tmp3));
            CKI(cub::DeviceRadixSort::SortPairs(d_tmp.p, tmp3, t[0].p, keys_out.p, perm_in.p, perm_out.p, (int)n_kept, 0, 64, e->stream));
            k5_keep_last_of_run<<<gk, 256, 0, e->stream>>>(keys_out.p, n_kept, d_keep.p);
            size_t tmp4 = 0;
            CKI(cub::DeviceScan::ExclusiveSum(nullptr, tmp4, d_keep.p, d_pos.p, n_kept, e->stream));
            CKI(d_tmp.ensure(tmp4));
            CKI(cub::DeviceScan::ExclusiveSum(d_tmp.p, tmp4, d_keep.p, d_pos.p, n_kept, e->stream));
            k5_gather_sorted<<<gk, 256, 0, e->stream>>>(tc, perm_out.p, d_keep.p, d_pos.p, n_kept, cur);
            CKI(cudaGetLastError());
            int32_t lp = 0, lk = 0;
            CKI(cudaMemcpyAsync(&lp, d_pos.p + (n_kept - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
            CKI(cudaMemcpyAsync(&lk, d_keep.p + (n_kept - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
            CKI(cudaStreamSynchronize(e->stream));
            n_kept = (int64_t)lp + lk;
            keys_out.release(); perm_in.release(); perm_out.release();
            h_scal[3] = 0;                                      // ascending now (NaN wavenumbers cannot get here: the range filter drops them)
        }
    } else {
        e->lines_set = false;
        int rc = alloc_line_storage(e, 0);
        if (rc) { cleanup(); return rc; }
    }
        lap("scatter + finalize");
#undef CKI
    cleanup();
    lap("free");
    if (h_scal[3] & 0xffffffffull) return fail(PRB_ERR_ARG, "prb_ingest_hitran_csv: wavenumbers are not ascending");
    double smax;
    memcpy(&smax, &h_scal[2], sizeof smax);
    e->n_lines = n_kept;
    e->n_groups = 1;
    e->has_group = false;
    e->s_max = smax;
    e->lines_set = true;
    e->grid_set = false;
    e->last.valid = false;
    if (n_lines_out) *n_lines_out = n_kept;
    return PRB_OK;
}

// Two-column xsc table text -> (wavenumber, cross section) arrays, parsed on the device like the line lists.
extern "C" int prb_parse_xsc_text(prb_engine *e, const char *text, int64_t n_bytes, int64_t capacity, double *wavenumber,
                                  double *cross_section, int64_t *n_rows_out) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n_bytes < 0 || (n_bytes > 0 && !text) || capacity < 0 || !n_rows_out || (capacity > 0 && (!wavenumber || !cross_section)))
        return fail(PRB_ERR_ARG, "prb_parse_xsc_text: bad arguments");
    if (n_bytes > (int64_t(1) << 31)) return fail(PRB_ERR_ARG, "prb_parse_xsc_text: more than 2 GiB of text");
    CK(cudaSetDevice(e->device));
    *n_rows_out = 0;
    if (n_bytes == 0) return PRB_OK;
    IngestScratch &g = e->ingest;
    const int64_t n_pad = std::max<int64_t>((n_bytes + 15) & ~int64_t(15), 16);
    CK(g.text.ensure(n_pad));
    CK(g.nl.ensure(n_pad));
    CK(g.scal.ensure(8));
    CK(cudaMemsetAsync(g.text.p + (n_pad - 16), 0, 16, e->stream));
    CK(cudaMemcpyAsync(g.text.p, text, n_bytes, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemsetAsync(g.scal.p, 0, 64, e->stream));
    k5_mark_newlines<<<(unsigned)((n_pad / 16 + 255) / 256), 256, 0, e->stream>>>(g.text.p, n_bytes, g.nl.p, g.scal.p);
    CK(cudaGetLastError());
    unsigned long long n_nl_u = 0;
    CK(cudaMemcpyAsync(&n_nl_u, g.scal.p, sizeof n_nl_u, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    const int64_t n_nl = (int64_t)n_nl_u;
    const int64_t n_rows = n_nl + (text[n_bytes - 1] != '\n' ? 1 : 0);
    if (n_rows == 0) return PRB_OK;
    CK(g.nlpos.ensure(n_nl + 1));
    size_t tmp_bytes = 0;
    thrust::counting_iterator<int64_t> counting(0);
    long long *d_selected = reinterpret_cast<long long *>(g.scal.p + 4);
    CK(cub::DeviceSelect::Flagged(nullptr, tmp_bytes, counting, g.nl.p, g.nlpos.p, d_selected, n_bytes, e->stream));
    CK(g.tmp.ensure(tmp_bytes));
    CK(cub::DeviceSelect::Flagged(g.tmp.p, tmp_bytes, counting, g.nl.p, g.nlpos.p, d_selected, n_bytes, e->stream));
    for (int c = 0; c < 4; ++c) CK(g.cols[c].ensure(n_rows));
    CK(g.keep.ensure(n_rows));
    CK(g.pos.ensure(n_rows + 1));
    k5_parse_xsc_rows<<<(unsigned)((n_rows + K5_ROWS - 1) / K5_ROWS), K5_ROWS, 0, e->stream>>>(g.text.p, n_bytes, g.nlpos.p, n_nl,
                                                                                             n_rows, g.cols[0].p, g.cols[1].p, g.keep.p);
    CK(cudaGetLastError());
    size_t tmp2 = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp2, g.keep.p, g.pos.p, n_rows, e->stream));
    CK(g.tmp.ensure(tmp2));
    CK(cub::DeviceScan::ExclusiveSum(g.tmp.p, tmp2, g.keep.p, g.pos.p, n_rows, e->stream));
    int32_t last_pos = 0, last_keep = 0;
    CK(cudaMemcpyAsync(&last_pos, g.pos.p + (n_rows - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(&last_keep, g.keep.p + (n_rows - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    const int64_t kept = (int64_t)last_pos + last_keep;
    *n_rows_out = kept;
    if (kept > capacity) return fail(PRB_ERR_ARG, "prb_parse_xsc_text: output capacity too small (n_rows_out holds the count)");
    if (kept == 0) return PRB_OK;
    k5_scatter2<<<(unsigned)((n_rows + 255) / 256), 256, 0, e->stream>>>(g.cols[0].p, g.cols[1].p, g.keep.p, g.pos.p, n_rows,
                                                                       g.cols[2].p, g.cols[3].p);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(wavenumber, g.cols[2].p, sizeof(double) * kept, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(cross_section, g.cols[3].p, sizeof(double) * kept, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return PRB_OK;
}

extern "C" int prb_download_lines(prb_engine *e, double *nu0, double *s296, double *einstein_a, double *elower,
                                  double *gamma_air, double *gamma_self, double *delta_air, double *n_air) {
    if (!e || !e->lines_set) return fail(PRB_ERR_STATE, "prb_download_lines: no line list on the device");
    CK(cudaSetDevice(e->device));
    const int64_t n = e->n_lines;
    double *dst[8] = {nu0, s296, einstein_a, elower, gamma_air, gamma_self, delta_air, n_air};
    const double *src[8] = {e->nu0.p, e->s296.p, e->einstein_a.p, e->elower.p, e->gair.p, e->gself.p, e->delta.p, e->nair.p};
    for (int c = 0; c < 8; ++c)
        if (dst[c] && n) CK(cudaMemcpyAsync(dst[c], src[c], sizeof(double) * n, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return PRB_OK;
}

extern "C" int64_t prb_line_count(prb_engine *e) { return (e && e->lines_set) ? e->n_lines : -1; }

// The number parser on the host (same source as the device kernel) for the CPU test suite.
extern "C" int prb_debug_parse_double(const char *text, int64_t n_bytes, double *value) {
    if (!text || !value || n_bytes < 0) return PRB_ERR_ARG;
    return parse_double(text, text + n_bytes, value) ? PRB_OK : PRB_ERR_PARSE;
}

// Zero-copy result delivery: the kernels that finish the spectra (K2's fused epilogue / K3) also store them into
// the caller's PINNED host buffers (TMA bulk stores over PCIe, tile by tile while the rest of the line sum runs),
// so when prb_atmosphere returns the results are already in host memory -- no separate device-to-host copy.
extern "C" int prb_set_result_host(prb_engine *e, float *radiance_host, float *transmittance_host, int64_t n_points) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (!radiance_host && !transmittance_host) {                  // switch off
        e->host_rad_dev = e->host_trans_dev = nullptr;
        e->host_result_len = 0;
        return PRB_OK;
    }
    if (!radiance_host || !transmittance_host || n_points < 1)
        return fail(PRB_ERR_ARG, "prb_set_result_host: both buffers and their length are required");
    if (((uintptr_t)radiance_host | (uintptr_t)transmittance_host) & 15)
        return fail(PRB_ERR_ARG, "prb_set_result_host: buffers must be 16-byte aligned");
    CK(cudaSetDevice(e->device));
    void *dr = nullptr, *dt = nullptr;
    if (cudaHostGetDevicePointer(&dr, radiance_host, 0) != cudaSuccess ||
        cudaHostGetDevicePointer(&dt, transmittance_host, 0) != cudaSuccess) {
        cudaGetLastError();
        return fail(PRB_ERR_ARG, "prb_set_result_host: buffers must be pinned host memory (cudaHostAlloc / cudaHostRegister / "
                                 "torch pin_memory); pageable memory cannot be written from the device");
    }
    e->host_rad_dev = (float *)dr;
    e->host_trans_dev = (float *)dt;
    e->host_result_len = n_points;
    return PRB_OK;
}

// ------------------------------------------------------------------------------------ gas cell, host to host, pipelined
// One call from HOST line columns to HOST spectra with the copies overlapped with the compute in both directions:
//   * the S296 column goes first (the FP32 scale of the records needs max|S|), then the other columns in S pieces,
//     wavenumber ascending, on a copy stream;
//   * the grid chunk is cut into S pieces of TWO WAVES of K2 tiles each (2 x 2 CTAs x SM count); piece s of the lines is
//     what sub-launch s needs beyond the earlier pieces (its tiles' windows plus margin), so K0/K1/K2 of piece s start
//     as soon as its lines have landed while the later pieces are still crossing PCIe;
//   * finished tiles leave through K2's fused epilogue: into the device result arrays, every peer's gather buffer
//     when connected, and the pinned host buffers registered with prb_set_result_host.
// The arithmetic is that of prb_upload_lines + prb_set_grid + prb_atmosphere(1 layer), bit for bit (same tiles, same
// records); narrow windows and tiny inputs simply take that sequence.
extern "C" int prb_gas_cell_host(prb_engine *e, int64_t n, const double *nu0, const double *s296, const double *gamma_air,
                                 const double *gamma_self, const double *elower, const double *n_air,
                                 const double *delta_air, const int32_t *group, int32_t n_groups, double range_min,
                                 double res, int64_t n_total, int64_t i_begin, int64_t i_end, double depth_cm,
                                 double t_layer, double p_layer, const double *conc, const double *molmass,
                                 const double *q_t, const double *q_296, int64_t window_len, double t_surface,
                                 double range_max) {
    if (!e) return fail(PRB_ERR_ARG, "null engine");
    if (n < 0 || n > 2000000000LL || n_groups < 1) return fail(PRB_ERR_ARG, "prb_gas_cell_host: bad line count / n_groups");
    if (n > 0 && (!nu0 || !s296 || !gamma_air || !gamma_self || !elower || !n_air || !delta_air))
        return fail(PRB_ERR_ARG, "prb_gas_cell_host: NULL column");
    if (!(res > 0) || n_total < 0 || i_begin < 0 || i_end < i_begin || i_end > n_total || n_total > 2000000000LL)
        return fail(PRB_ERR_ARG, "prb_gas_cell_host: bad grid");
    if (!conc || !molmass || !q_t || !q_296 || window_len < 1) return fail(PRB_ERR_ARG, "prb_gas_cell_host: bad layer arguments");
    CK(cudaSetDevice(e->device));
    const int64_t nc = i_end - i_begin;
    const int64_t wm = std::max<int64_t>(window_len - 2, 0);
    const int ppt = pick_ppt(e, wm);
    const int tile_pts = K2_CONSUMERS * 32 * ppt;
    const int n_tiles = (int)((nc + tile_pts - 1) / tile_pts);
    // K2 tiles per piece in waves of resident CTAs: measured on cfg2 (ms per call) 1 wave 1.72, 2 waves 1.65, 3 waves 1.65.
    // The FIRST piece is a single wave: its lines are across PCIe in half the time, so the first line sum starts earlier
    // while the second piece still lands under it (PRB_PIPE_FIRST_WAVES).
#ifndef PRB_PIPE_FIRST_WAVES
#define PRB_PIPE_FIRST_WAVES 1
#endif
    const int waves_per_piece = 2;
    const int wave1 = K2_MIN_CTAS * e->prop.multiProcessorCount;
    const int wave = waves_per_piece * wave1;
    const int first = std::min(n_tiles, PRB_PIPE_FIRST_WAVES * wave1);
    const int S = (first > 0 ? 1 : 0) + (n_tiles - first + wave - 1) / wave;
    // (per-layer line ranges and a continuum: the separate calls apply them)
    const bool pipelined = k2_classed(e) && e->fuse_single && wm >= e->narrow_wm && S >= 2 && n >= 4096 && e->line_lo.empty() &&
                           e->cont_tab.empty();
    if (!pipelined) {
        int rc = prb_upload_lines(e, n, nu0, s296, gamma_air, gamma_self, elower, n_air, delta_air, group, n_groups);
        if (rc) return rc;
        if ((rc = prb_set_grid(e, range_min, res, n_total, i_begin, i_end))) return rc;
        return prb_atmosphere(e, 1, n_groups, &depth_cm, &t_layer, &p_layer, conc, molmass, q_t, q_296, &window_len,
                              t_surface, range_max);
    }
    if (nc + 2 * wm + 8192 >= (int64_t(1) << 24))
        return fail(PRB_ERR_RANGE, "owned grid chunk plus cutoff windows exceeds 2^24 points; shard the grid");
    if (!e->copy_stream) {
        CK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&e->stream2, cudaStreamNonBlocking));
        if (!e->pin_scal) CK(cudaMallocHost((void **)&e->pin_scal, 64));
        CK(e->dev_scal.ensure(8));
    }
    while ((int)e->pipe_ev.size() < 2 * (S + 1)) {
        cudaEvent_t x;
        CK(cudaEventCreateWithFlags(&x, cudaEventDisableTiming));
        e->pipe_ev.push_back(x);
    }
    e->lines_set = false;
    e->grid_set = false;
    e->last.valid = false;
    int rc = alloc_line_storage(e, n);
    if (rc) return rc;
    e->n_lines = n;
    e->n_groups = n_groups;
    e->has_group = group != nullptr;
    if (group) CK(e->group.ensure(e->n_alloc));
    e->range_min = range_min; e->res = res; e->n_total = n_total; e->i_begin = i_begin; e->i_end = i_end;

    // S296 first: max|S| fixes the power-of-two scale of every record
    CK(cudaMemsetAsync(e->dev_scal.p, 0, 64, e->stream));
    CK(cudaEventRecord(e->pipe_ev[S], e->stream));
    CK(cudaStreamWaitEvent(e->copy_stream, e->pipe_ev[S], 0));
    CK(cudaMemcpyAsync(e->s296.p, s296, sizeof(double) * n, cudaMemcpyHostToDevice, e->copy_stream));
    CK(cudaEventRecord(e->pipe_ev[S], e->copy_stream));
    CK(cudaStreamWaitEvent(e->stream, e->pipe_ev[S], 0));
    k0_absmax<<<e->prop.multiProcessorCount * 4, 256, 0, e->stream>>>(e->s296.p, n, e->dev_scal.p);
    CK(cudaGetLastError());

    // piece boundaries: sub-launch s owns tiles [s*wave, (s+1)*wave) and needs the lines whose grid index lies in
    // [first point - wm, last point + wm]; two grid points of slack cover the truncation of the index
    UploadPipe pipe;
    pipe.S = S;
    pipe.ev.assign(e->pipe_ev.begin(), e->pipe_ev.begin() + S);
    pipe.ev_k1.assign(e->pipe_ev.begin() + S + 1, e->pipe_ev.begin() + 2 * (S + 1));
    pipe.stream2 = e->stream2;
    pipe.smax_bits_dev = e->dev_scal.p;
    pipe.scale_dev = reinterpret_cast<double *>(e->dev_scal.p + 2);
    for (int sidx = 0; sidx < S; ++sidx) {
        const int t0 = sidx == 0 ? 0 : first + (sidx - 1) * wave, t1 = sidx == 0 ? first : std::min(n_tiles, t0 + wave);
        const int64_t p0 = (int64_t)t0 * tile_pts, p1 = std::min<int64_t>(nc, (int64_t)t1 * tile_pts);
        const double nu_lo = range_min + (double)(i_begin + p0 - wm - 2) * res;
        const double nu_hi = range_min + (double)(i_begin + p1 - 1 + wm + 3) * res;
        int64_t lo = std::lower_bound(nu0, nu0 + n, nu_lo) - nu0;
        int64_t hi = sidx == S - 1 ? n : std::upper_bound(nu0, nu0 + n, nu_hi) - nu0;
        if (sidx && hi < pipe.line_hi[sidx - 1]) hi = pipe.line_hi[sidx - 1];
        if (lo > hi) lo = hi;
        pipe.tile_lo.push_back(t0);
        pipe.tile_hi.push_back(t1);
        pipe.line_lo.push_back(lo);
        pipe.line_hi.push_back(hi);
    }
    // the other columns, piece by piece, on the copy stream (piece 0 now, piece s+1 while piece s is being launched)
    DevBuf<double> *cols[6] = {&e->nu0, &e->gair, &e->gself, &e->elower, &e->nair, &e->delta};
    const double *src[6] = {nu0, gamma_air, gamma_self, elower, n_air, delta_air};
    pipe.enqueue_piece = [&](int sidx) -> int {
        const int64_t a = sidx ? pipe.line_hi[sidx - 1] : 0, b = pipe.line_hi[sidx];
        if (b > a) {
            for (int c = 0; c < 6; ++c)
                CK(cudaMemcpyAsync(cols[c]->p + a, src[c] + a, sizeof(double) * (b - a), cudaMemcpyHostToDevice, e->copy_stream));
            if (group)
                CK(cudaMemcpyAsync(e->group.p + a, group + a, sizeof(int32_t) * (b - a), cudaMemcpyHostToDevice, e->copy_stream));
        }
        CK(cudaEventRecord(e->pipe_ev[sidx], e->copy_stream));
        return PRB_OK;
    };
    if ((rc = pipe.enqueue_piece(0))) return rc;

    rc = atmosphere_impl(e, 1, n_groups, &depth_cm, &t_layer, &p_layer, conc, molmass, q_t, q_296, &window_len, t_surface,
                         range_max, &pipe);
    // what prb_upload_lines checks before it returns, checked here after the fact (the header says so: on
    // PRB_ERR_ARG from this check the output buffers hold garbage)
    k0_validate_lines<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(e->nu0.p, group ? e->group.p : nullptr, n, n_groups,
                                                                        reinterpret_cast<unsigned int *>(e->dev_scal.p + 1));
    cudaMemcpyAsync(e->pin_scal, e->dev_scal.p, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream);
    CK(cudaStreamSynchronize(e->copy_stream));
    CK(cudaStreamSynchronize(e->stream2));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
    if (rc) return rc;                                          // a failed launch sequence: its own message stands
    memcpy(&e->s_max, e->pin_scal, sizeof(double));             // max|S296|, for the planning of later calls
    const unsigned int vf = (unsigned int)e->pin_scal[1];
    if (vf & 1u) return fail(PRB_ERR_ARG, "prb_gas_cell_host: nu0 must be ascending");
    if (vf & 2u) return fail(PRB_ERR_ARG, "prb_gas_cell_host: group id out of range");
    e->lines_set = true;
    e->grid_set = true;
    return PRB_OK;
}
