// k3_stream.cuh -- K3: fused pointwise layer physics (HBM-bound streaming kernels).
//
//   absCoef        pyradClasses.py:581-583, 707-712   k = sum_m sigma_m * (conc_m P / 1e4 / kB / T)
//   transmittance  pyradClasses.py:585-587, 714-716   T = exp(-k * depth)
//   Planck         pyradPlanck.py:38-44, 12-15        B = 2e8 h c^2 nu^3 / (exp(100 h c nu / kB / T) - 1)
//   transmission   pyradClasses.py:784-787            I_out = T * I_in + (1 - T) * B(nu, T_layer)
//   xsc ingest     pyradClasses.py:159-162, 493-500   np.interp + aligned placement
//   multi-layer    fold of Layer.transmission over the layers (absent upstream, SURVEY 3.5)
//
// Two flavours: an FP64 kernel behind the host-buffer API (bit-faithful formulas, used by the
// pyradClasses mirror), and the FP32 float4-vectorised fold over the resident k matrix used by
// the atmosphere path (algorithmic traffic L*N*4 + N*8 bytes).
#pragma once
#include "common.cuh"

namespace prb {

// nu_i of np.linspace(start, stop, n): i*step + start (two roundings, as numpy), last = stop.  The host evaluates the
// same two roundings (no FMA contraction) when it turns band edges into point indices.
__host__ __device__ __forceinline__ double axis_value(int64_t i, int64_t n, double x0, double dx, double x_last) {
    if (i == n - 1) return x_last;
#ifdef __CUDA_ARCH__
    return __dadd_rn(__dmul_rn((double)i, dx), x0);
#else
    volatile double p = (double)i * dx;                // a separate rounding of the product, as __dmul_rn
    return p + x0;
#endif
}

__device__ __forceinline__ double planck_f64(double nu, double temp) {
    const double a = 2E8 * hPlanck * (cLight * cLight) * (nu * nu * nu);
    const double b = 100 * hPlanck * cLight * nu / kBoltz / temp;
    return a / (exp(b) - 1);                              // nu = 0 -> 0/0 = NaN, as the reference
}

__global__ void __launch_bounds__(256)
k3_layer_stream_f64(int64_t n, int n_mol, const double *__restrict__ sigma, const double *__restrict__ weight,
                    double depth, double t_layer, double x0, double dx, double x_last,
                    const double *__restrict__ rad_in, double *__restrict__ absc, double *__restrict__ trans,
                    double *__restrict__ rad_out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double k = 0.0;
        for (int m = 0; m < n_mol; ++m) k += sigma[(int64_t)m * n + i] * weight[m];
        const double t = exp(-k * depth);
        if (absc) absc[i] = k;
        if (trans) trans[i] = t;
        if (rad_out) {
            const double b = planck_f64(axis_value(i, n, x0, dx, x_last), t_layer);
            rad_out[i] = t * rad_in[i] + (1 - t) * b;
        }
    }
}

// The same layer physics on rows that are already on the device: the per-group cross sections of the last
// prb_line_sum_groups (rows_a) and the resident xsc tables (rows_b), on the owned chunk [i_first, i_first + n) of a grid
// of n_total points.  k = sum_a sigma_a w_a + sum_b sigma_b w_b, in that order (Layer.absCoef, pyradClasses.py:707-712).
__global__ void __launch_bounds__(256)
k3_layer_stream_rows_f64(int64_t n, int n_a, const double *__restrict__ rows_a, int64_t ld_a,
                         const double *__restrict__ w_a, int n_b, const double *__restrict__ rows_b, int64_t ld_b,
                         const double *__restrict__ w_b, double depth, double t_layer, int64_t i_first, int64_t n_total,
                         double x0, double dx, double x_last, const double *__restrict__ rad_in,
                         double *__restrict__ absc, double *__restrict__ trans, double *__restrict__ rad_out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double k = 0.0;
        for (int m = 0; m < n_a; ++m) k += rows_a[(int64_t)m * ld_a + i] * w_a[m];
        for (int m = 0; m < n_b; ++m) k += rows_b[(int64_t)m * ld_b + i] * w_b[m];
        const double t = exp(-k * depth);
        if (absc) absc[i] = k;
        if (trans) trans[i] = t;
        if (rad_out) {
            const double b = planck_f64(axis_value(i_first + i, n_total, x0, dx, x_last), t_layer);
            rad_out[i] = t * rad_in[i] + (1 - t) * b;
        }
    }
}

__global__ void __launch_bounds__(256)
k3_planck_f64(int64_t n, double x0, double dx, double x_last, double temp, double *__restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = planck_f64(axis_value(i, n, x0, dx, x_last), temp);
}

// np.interp(x, xp, fp) for one x: clamps outside, slope form inside (numpy's arithmetic, no FMA).
__device__ __forceinline__ double np_interp(double x, const double *__restrict__ xp, const double *__restrict__ fp,
                                            int64_t n) {
    if (x <= xp[0]) return x < xp[0] ? fp[0] : fp[0];
    if (x >= xp[n - 1]) return fp[n - 1];
    int64_t lo = 0, hi = n - 1;                            // xp[lo] <= x < xp[hi]
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (xp[mid] <= x) lo = mid; else hi = mid;
    }
    const double slope = __ddiv_rn(__dsub_rn(fp[lo + 1], fp[lo]), __dsub_rn(xp[lo + 1], xp[lo]));
    return __dadd_rn(__dmul_rn(slope, __dsub_rn(x, xp[lo])), fp[lo]);
}

// out[0 .. n_out) holds the grid points [i_first, i_first + n_out) of the placement (i_first = 0: the whole grid; the
// resident tables of the atmosphere path are built for the owned chunk only).
__global__ void __launch_bounds__(256)
k3_xsc_place(int64_t n_out, int64_t dst0, int64_t src0, int64_t count, int interp, double ax0, double adelta,
             int64_t n_file, const double *__restrict__ fx, const double *__restrict__ fy, double *__restrict__ out,
             int64_t i_first) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_out; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t j = i_first + i - dst0;
        double v = 0.0;
        if (j >= 0 && j < count) {
            const int64_t m = src0 + j;
            if (interp) v = np_interp(__dadd_rn(ax0, __dmul_rn((double)m, adelta)), fx, fy, n_file);
            else v = (m >= 0 && m < n_file) ? fy[m] : 0.0;
        }
        out[i] = v;
    }
}

constexpr int K3_UNROLL = 8;

// Optical depth of the whole column: the per-layer terms -tau_l log2(e) are summed in FP32 over groups of
// K3_TAU_GROUP consecutive layers (aligned to the layer index, so every fold kernel forms the same groups) and the
// group sums are added into a double-float (hi, lo) pair with an error-free TwoSum.  A plain FP32 running sum over
// 100 layers loses up to ~100 * 2^-24 of tau, i.e. up to 2e-6 of the total transmittance at tau ~ 1 -- more than the
// 1e-6 the path promises; this way the error stays below 4 * 2^-24 * tau (|dT| <= 9e-8) for six FP32 instructions per
// point per four layers (FP64 accumulators would cost the fold kernel eight registers it does not have).
constexpr int K3_TAU_GROUP = 4;
__device__ __forceinline__ void tau_flush(float (&tau)[4], float (&hi)[4], float (&lo)[4]) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float s = __fadd_rn(hi[q], tau[q]);
        const float bp = __fsub_rn(s, hi[q]);
        const float err = __fadd_rn(__fsub_rn(hi[q], __fsub_rn(s, bp)), __fsub_rn(tau[q], bp));
        lo[q] = __fadd_rn(lo[q], err);
        hi[q] = s;
        tau[q] = 0.f;
    }
}

// ---- atmosphere fold, FP32 storage, float4 per thread --------------------------------------------
struct FoldLayer {
    float neg_depth_log2e;   // -depth * log2(e): T = exp2(k * this)
    float c2_over_t;         // 100 h c / kB / T_layer
};

__device__ __forceinline__ float k3_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float k3_ex2(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

__device__ __forceinline__ float planck_f32(float a_nu3, float x) {
    // a nu^3 / (e^x - 1), x = c2 nu / T, to ~1e-7 relative with as few MUFU operations as the range allows:
    //   x >  8.5 : y = e^-x < 2.1e-4, 1/(e^x - 1) = y/(1 - y) = y + y^2 + O(y^3)       -- one MUFU (ex2)
    //   x >= .25 : rcp(e^x - 1)                                                        -- two MUFU (ex2, rcp)
    //   x <  .25 : the subtraction cancels, so the first few hundred grid points (nu < ~40 cm^-1) take expm1f.
    if (x > 8.5f) {
        const float y = k3_ex2(x * -1.4426950408889634f);
        return a_nu3 * fmaf(y, y, y);
    }
    if (x < 0.25f) return a_nu3 / expm1f(x);
    return a_nu3 * k3_rcp(k3_ex2(x * 1.4426950408889634f) - 1.0f);
}

// One layer of the fold: I <- T I + (1 - T) B with T = 2^e, e = -tau log2(e).  Two evaluation orders, chosen per
// point and layer: where the layer is optically thin (|e| < 1/8, T > 0.917) the emission weight 1 - T comes from the
// series of -expm1(e ln 2) and the update is I + (1 - T)(B - I); elsewhere it is B + T (I - B).  With T alone the
// thin case computes 1 - T by cancellation from a MUFU.EX2 result that is good to ~1e-7 ABSOLUTE: a warm, nearly
// transparent layer above a cold opaque one (the stratopause seen at 4000 cm^-1: B_layer = 300 I, tau = 1e-4) then
// adds 300 * 1e-7 of I per layer, all of one sign -- 2.5e-5 of the radiance after 30 such layers (measured against
// the oracle at full size, tests/test_gpu_fullsize.py).  The thick-layer form must stay for T -> 0: I + (B - I)
// would round at the size of I, not of B.  Series: five terms, truncation below 7e-9 of 1 - T at |e| = 1/8.
__device__ __forceinline__ float k3_fold_step(float rad, float e, float b) {
    const float t = k3_ex2(e);
    // 1 - 2^e = -e (c1 + e (c2 + e (c3 + e (c4 + e c5)))),  c_n = ln(2)^n / n!
    float p = fmaf(e, 1.3333558146e-3f, 9.6181291076e-3f);
    p = fmaf(e, p, 5.5504108665e-2f);
    p = fmaf(e, p, 2.4022650696e-1f);
    p = fmaf(e, p, 6.9314718056e-1f);
    const bool thin = fabsf(e) < 0.125f;
    const float d = rad - b;
    return thin ? fmaf(e * p, d, rad) : fmaf(t, d, b);     // thin: I - (1 - T)(I - B), (1 - T) = -e p
}

// The same step for two points at once with Blackwell's packed FP32x2 instructions (the fold is issue bound: half the
// instructions for the multiply, the series, the difference, both candidate updates).  Lane for lane the operations and
// their roundings are those of k3_fold_step, so the two agree bit for bit.
__device__ __forceinline__ float2 k3_fold_step2(float2 rad, float2 e, float2 b) {
    const float2 t = make_float2(k3_ex2(e.x), k3_ex2(e.y));
    float2 p = __ffma2_rn(e, make_float2(1.3333558146e-3f, 1.3333558146e-3f), make_float2(9.6181291076e-3f, 9.6181291076e-3f));
    p = __ffma2_rn(e, p, make_float2(5.5504108665e-2f, 5.5504108665e-2f));
    p = __ffma2_rn(e, p, make_float2(2.4022650696e-1f, 2.4022650696e-1f));
    p = __ffma2_rn(e, p, make_float2(6.9314718056e-1f, 6.9314718056e-1f));
    const float2 d = __ffma2_rn(b, make_float2(-1.f, -1.f), rad);              // rad - b, one rounding
    const float2 thin = __ffma2_rn(__fmul2_rn(e, p), d, rad);
    const float2 thick = __ffma2_rn(t, d, b);
    return make_float2(fabsf(e.x) < 0.125f ? thin.x : thick.x, fabsf(e.y) < 0.125f ? thin.y : thick.y);
}

// Destinations of the finished spectra: this rank's slot in every rank's gather buffer (peer memory over
// NVLink; stores are fire-and-forget), or just the local result arrays when no peers are connected.
constexpr int K3_MAX_PEERS = 8;
constexpr int K3_MAX_DST = K3_MAX_PEERS + 1;          // + the caller's pinned host result buffers (zero-copy)
struct K3Dst {
    int n;
    float *rad[K3_MAX_DST];
    float *trans[K3_MAX_DST];
};

__global__ void __launch_bounds__(256)
k3_fold_f32(const float *__restrict__ kmat, int64_t ld, int n_layers, const FoldLayer *__restrict__ layers,
            int64_t n_chunk, int64_t i_begin, int64_t n_total, double x0, double dx, double x_last,
            float c2_over_tsurf, const K3Dst dst) {
    const int64_t nvec = (n_chunk + 3) >> 2;
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i0 = v << 2;
        float nu[4], a3[4], rad[4], tau[4];
        float tau_hi[4], tau_lo[4];                              // optical depth of the column, see K3_TAU_GROUP
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double x = axis_value(i_begin + i0 + q, n_total, x0, dx, x_last);
            nu[q] = (float)x;
            a3[q] = (float)(2E8 * hPlanck * (cLight * cLight) * (x * x * x));
            rad[q] = planck_f32(a3[q], c2_over_tsurf * nu[q]);   // I_0 = B(nu, T_surface)
            tau[q] = 0.f;
            tau_hi[q] = 0.f;
            tau_lo[q] = 0.f;
        }
        // layers in groups of K3_UNROLL: all of a group's loads are issued before its math, so every thread keeps
        // K3_UNROLL x 16 B in flight (the kernel is latency bound otherwise); the k matrix is read exactly once,
        // hence the streaming (evict-first) loads.
        const float *col = kmat + i0;
        for (int l0 = 0; l0 < n_layers; l0 += K3_UNROLL) {
            float4 k4[K3_UNROLL];
#pragma unroll
            for (int j = 0; j < K3_UNROLL; ++j)
                k4[j] = (l0 + j < n_layers) ? __ldcs(reinterpret_cast<const float4 *>(col + (int64_t)(l0 + j) * ld))
                                            : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int j = 0; j < K3_UNROLL; ++j) {
                if (l0 + j < n_layers) {
                    const FoldLayer fl = layers[l0 + j];
                    const float kk[4] = {k4[j].x, k4[j].y, k4[j].z, k4[j].w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float e = kk[q] * fl.neg_depth_log2e;       // -tau_l * log2(e)
                        const float b = planck_f32(a3[q], fl.c2_over_t * nu[q]);
                        rad[q] = k3_fold_step(rad[q], e, b);              // T*I + (1-T)*B
                        tau[q] += e;
                    }
                    if (((l0 + j) & (K3_TAU_GROUP - 1)) == K3_TAU_GROUP - 1) tau_flush(tau, tau_hi, tau_lo);
                }
            }
        }
        tau_flush(tau, tau_hi, tau_lo);
        const float4 r4 = make_float4(rad[0], rad[1], rad[2], rad[3]);
        const float4 t4 = make_float4(exp2f(tau_hi[0] + tau_lo[0]), exp2f(tau_hi[1] + tau_lo[1]), exp2f(tau_hi[2] + tau_lo[2]),
                                      exp2f(tau_hi[3] + tau_lo[3]));
        const float rr[4] = {r4.x, r4.y, r4.z, r4.w}, tt[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll 1
        for (int d = 0; d < dst.n; ++d) {
            if (i0 + 3 < n_chunk) {
                *reinterpret_cast<float4 *>(dst.rad[d] + i0) = r4;
                *reinterpret_cast<float4 *>(dst.trans[d] + i0) = t4;
            } else {
                for (int q = 0; q < 4 && i0 + q < n_chunk; ++q) {
                    dst.rad[d][i0 + q] = rr[q];
                    dst.trans[d][i0 + q] = tt[q];
                }
            }
        }
    }
}

// ---- the same fold with the k matrix staged through shared memory by TMA ----------------------------------------
// A CTA owns strips of 1024 grid points (one float4 per thread) and walks the layers in groups of K3T_LAYERS rows:
// one elected thread issues a bulk copy per row (4 KB each) into a small ring, one group ahead of the math, so the
// loads in flight (5 CTAs x 16 KB per SM) are not held in registers; the math reads its float4 from shared memory
// (conflict free).  Ring geometry measured on B200 (rows:slots:CTAs/SM -> ms at cfg4): 4:2:5 0.406, 4:3:4 0.424,
// 6:3:3 0.459, 4:4:3 0.463, 2:4:6 0.535, 8:3:2 0.537.  The fold is instruction bound rather than memory bound (measured: staging alone
// changes nothing), so above nu_interp_min the layer's Planck term is evaluated at the thread's first and last point
// only and interpolated linearly for the two between -- half the instructions per point; k3_fold_f32 keeps the
// per-point evaluation and is the reference the tests compare against.
constexpr int K3T_THREADS = 256;
constexpr int K3T_STRIP = K3T_THREADS * 4;             // points per strip
#ifndef PRB_K3T_LAYERS
#define PRB_K3T_LAYERS 4
#endif
#ifndef PRB_K3T_SLOTS
#define PRB_K3T_SLOTS 2
#endif
#ifndef PRB_K3T_MINB
#define PRB_K3T_MINB 5
#endif
constexpr int K3T_LAYERS = PRB_K3T_LAYERS;             // rows per ring slot
constexpr int K3T_SLOTS = PRB_K3T_SLOTS;
constexpr int K3T_MINB = PRB_K3T_MINB;                 // resident CTAs per SM the shared memory is sized for

// B(nu, T_l) at a thread's four consecutive points for one layer.  interp: evaluated at the first and last point only,
// the two between by linear interpolation (relative error < 1e-7 above the host's nu_interp_min, chosen from the grid
// spacing; one path decision per thread instead of per point); otherwise per point.  Shared by k3_fold_tma and
// k3_flux_tma, so a flux pass with mu = 1 reproduces the fold bit for bit.
__device__ __forceinline__ void k3_planck4(const float (&nu)[4], const float (&a3)[4], float c2_over_t, bool interp,
                                           float (&b)[4]) {
    if (interp) {
        const float xa = c2_over_t * nu[0], xb = c2_over_t * nu[3];
        float ba, bb;
        if (xa > 8.5f) {
            const float ya = k3_ex2(xa * -1.4426950408889634f), yb = k3_ex2(xb * -1.4426950408889634f);
            ba = a3[0] * fmaf(ya, ya, ya);
            bb = a3[3] * fmaf(yb, yb, yb);
        } else {
            ba = a3[0] * k3_rcp(k3_ex2(xa * 1.4426950408889634f) - 1.0f);
            bb = a3[3] * k3_rcp(k3_ex2(xb * 1.4426950408889634f) - 1.0f);
        }
        const float db = bb - ba;
        b[0] = ba; b[1] = fmaf(db, 1.0f / 3.0f, ba); b[2] = fmaf(db, 2.0f / 3.0f, ba); b[3] = bb;
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) b[q] = planck_f32(a3[q], c2_over_t * nu[q]);
    }
}

struct K3TSmem {
    float k[K3T_SLOTS][K3T_LAYERS][K3T_STRIP];
    float2 tau[4][K3T_THREADS];            // (hi, lo) optical-depth accumulators of every thread's four points
    uint64_t full[K3T_SLOTS];
};

__global__ void __launch_bounds__(K3T_THREADS, K3T_MINB)
k3_fold_tma(const float *__restrict__ kmat, int64_t ld, int n_layers, const FoldLayer *__restrict__ layers,
            int64_t n_chunk, int64_t i_begin, int64_t n_total, double x0, double dx, double x_last,
            float c2_over_tsurf, float nu_interp_min, const K3Dst dst) {
    extern __shared__ __align__(128) unsigned char k3_smem_raw[];
    K3TSmem &sm = *reinterpret_cast<K3TSmem *>(k3_smem_raw);
    const int tid = threadIdx.x;
    const int64_t n_strips = (n_chunk + K3T_STRIP - 1) / K3T_STRIP;
    const int groups = (n_layers + K3T_LAYERS - 1) / K3T_LAYERS;
    // the CTA's work as one flat sequence of (strip, layer group) steps
    const int64_t my_strips = blockIdx.x < n_strips ? (n_strips - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t n_steps = my_strips * groups;
    if (tid == 0) {
        for (int s = 0; s < K3T_SLOTS; ++s) mbar_init(&sm.full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    auto issue = [&](int64_t step) {                   // thread 0 only
        const int slot = (int)(step % K3T_SLOTS);
        const int64_t strip = blockIdx.x + (step / groups) * gridDim.x;
        const int g = (int)(step % groups);
        const int64_t p0 = strip * K3T_STRIP;
        const int64_t pts = min((int64_t)K3T_STRIP, ((n_chunk - p0) + 3) & ~int64_t(3));   // rows are padded to 4 floats
        const int rows = min(K3T_LAYERS, n_layers - g * K3T_LAYERS);
        mbar_expect_tx(&sm.full[slot], (uint32_t)(rows * pts * 4));
        for (int r = 0; r < rows; ++r)
            tma_bulk_g2s(sm.k[slot][r], kmat + (int64_t)(g * K3T_LAYERS + r) * ld + p0, (uint32_t)(pts * 4), &sm.full[slot]);
    };
    if (tid == 0)
        for (int64_t s = 0; s < min(n_steps, (int64_t)(K3T_SLOTS - 1)); ++s) issue(s);

    float nu[4], a3[4], rad[4], tau[4];
    // the column's (hi, lo) optical depth lives in shared memory, touched once per K3_TAU_GROUP layers: the register
    // budget of 5 CTAs per SM (48) has no room for it
    auto tau_flush_smem = [&]() {
        float hi[4], lo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) { const float2 v = sm.tau[q][tid]; hi[q] = v.x; lo[q] = v.y; }
        tau_flush(tau, hi, lo);
#pragma unroll
        for (int q = 0; q < 4; ++q) sm.tau[q][tid] = make_float2(hi[q], lo[q]);
    };
    bool interp = false;
    int64_t i0 = 0;
    for (int64_t step = 0; step < n_steps; ++step) {
        const int slot = (int)(step % K3T_SLOTS);
        const int g = (int)(step % groups);
        if (g == 0) {                                  // a new strip: surface radiance, zero optical depth
            const int64_t strip = blockIdx.x + (step / groups) * gridDim.x;
            i0 = strip * K3T_STRIP + 4 * tid;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double x = axis_value(i_begin + i0 + q, n_total, x0, dx, x_last);
                nu[q] = (float)x;
                a3[q] = (float)(2E8 * hPlanck * (cLight * cLight) * (x * x * x));
                rad[q] = planck_f32(a3[q], c2_over_tsurf * nu[q]);
                tau[q] = 0.f;
                sm.tau[q][tid] = make_float2(0.f, 0.f);
            }
            interp = nu[0] >= nu_interp_min;
        }
        // keep the ring two steps ahead: the slot being refilled was released by the barrier at the end of step-1
        if (tid == 0 && step + K3T_SLOTS - 1 < n_steps) issue(step + K3T_SLOTS - 1);
        mbar_wait(&sm.full[slot], (uint32_t)((step / K3T_SLOTS) & 1));
        const int rows = min(K3T_LAYERS, n_layers - g * K3T_LAYERS);
        if (i0 < n_chunk) {
#pragma unroll
            for (int r = 0; r < K3T_LAYERS; ++r) {
                if (r < rows) {
                    const float4 k4 = *reinterpret_cast<const float4 *>(&sm.k[slot][r][4 * tid]);
                    const FoldLayer fl = layers[g * K3T_LAYERS + r];
                    const float kk[4] = {k4.x, k4.y, k4.z, k4.w};
                    float b[4];
                    k3_planck4(nu, a3, fl.c2_over_t, interp, b);
                    {
                        const float2 nd = make_float2(fl.neg_depth_log2e, fl.neg_depth_log2e);
                        const float2 e01 = __fmul2_rn(make_float2(kk[0], kk[1]), nd), e23 = __fmul2_rn(make_float2(kk[2], kk[3]), nd);
                        const float2 r01 = k3_fold_step2(make_float2(rad[0], rad[1]), e01, make_float2(b[0], b[1]));
                        const float2 r23 = k3_fold_step2(make_float2(rad[2], rad[3]), e23, make_float2(b[2], b[3]));
                        const float2 t01 = __fadd2_rn(make_float2(tau[0], tau[1]), e01), t23 = __fadd2_rn(make_float2(tau[2], tau[3]), e23);
                        rad[0] = r01.x; rad[1] = r01.y; rad[2] = r23.x; rad[3] = r23.y;
                        tau[0] = t01.x; tau[1] = t01.y; tau[2] = t23.x; tau[3] = t23.y;
                    }
                    if (((g * K3T_LAYERS + r) & (K3_TAU_GROUP - 1)) == K3_TAU_GROUP - 1) tau_flush_smem();
                }
            }
        }
        __syncthreads();                               // every thread is done with this slot: it may be refilled
        if (g == groups - 1 && i0 < n_chunk) {
            tau_flush_smem();
            float tt4[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) { const float2 v = sm.tau[q][tid]; tt4[q] = exp2f(v.x + v.y); }
            const float4 r4 = make_float4(rad[0], rad[1], rad[2], rad[3]);
            const float4 t4 = make_float4(tt4[0], tt4[1], tt4[2], tt4[3]);
            const float rr[4] = {r4.x, r4.y, r4.z, r4.w}, tt[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll 1
            for (int d = 0; d < dst.n; ++d) {
                if (i0 + 3 < n_chunk) {
                    *reinterpret_cast<float4 *>(dst.rad[d] + i0) = r4;
                    *reinterpret_cast<float4 *>(dst.trans[d] + i0) = t4;
                } else {
                    for (int q = 0; q < 4 && i0 + q < n_chunk; ++q) {
                        dst.rad[d][i0 + q] = rr[q];
                        dst.trans[d][i0 + q] = tt[q];
                    }
                }
            }
        }
    }
}

// ---- flux fold: hemispheric fluxes and slant radiances over the resident k matrix --------------------------------
// For every node mu_i (NMU of them, 1..4) of a caller's angular quadrature, the fold I <- T I + (1 - T) B(nu, T_l) with
// T = exp(-k_l depth_l / mu_i) runs upward from I = B(nu, T_surface) at level 0 (DOWN = false), or downward from I = 0 at
// level L (DOWN = true).  Level j is the boundary below layer j: 0 = surface, L = top of the atmosphere.  The strips, the
// TMA ring and the Planck policy are k3_fold_tma's; B(nu, T_l) is evaluated once per point and layer and serves every
// node.  At each level a thread forms sum_i w_i mu_i sum_q I_i(nu_q) over its four points in FP32 (a value that is not
// finite counts as 0, see `partial`), a fixed xor-butterfly adds the warp's 32 values, and lane 0 adds the result into a per-(warp,
// level) FP64 accumulator in shared memory that lives for all of the CTA's strips.  The CTA then writes its per-level
// partials (warps in order) and k3_flux_sum adds them in CTA order: the result is deterministic, with no atomics.
//
// Band pass (BAND = true, prb_atmosphere_band_fluxes): the same fold, but each warp's sums are kept apart by wavenumber
// band instead of running over strips.  The 128 points of a warp (its span) meet zero or more bands; a segment is the
// intersection of a span with a band, numbered in position order (so a band's segments are consecutive).  At each level a
// span that lies inside one band forms exactly the sum above (partial() and the butterfly); a span that meets band edges
// forms one masked sum per segment (same non-finite rule) with the same butterfly.  Lane 0 stores each as FP64 into
// part[level][segment].  The CTA walks the host's list of strips that meet a band, and k3_flux_band_sum adds each band's
// segments in position order with a tree whose shape depends only on their count: the result depends on the edges and
// the span positions only, not on the launch grid.
//
// Boundaries (BOUND = true, prb_set_flux_boundaries): only the start values of the two passes change.  The downward pass
// starts from B(nu, T_top) at level L (0 when T_top = 0) and adds that level's sum.  It runs first and writes its surface
// rows.  The upward pass starts each strip from eps B(nu, T_s) + (1 - eps) S_i, S_i the radiance the surface reflects
// along mu_i: Lambertian S = sum_j 2 w_j mu_j I_down_j(nu, 0) (FP32, node order), specular S_i = I_down_i(nu, 0).  Where
// eps = 1 the start is B(nu, T_s) bit for bit, whatever comes down.  The layer loop is the fold's.
//
// Solar beam (SUN != K3F_NO_SUN, prb_set_solar_source; always with BOUND): a collimated beam E along mu_sun that nothing
// emits into or scatters.  The downward pass (SUN = K3F_SUN) carries E next to the nodes from E = S(nu) at level L,
// E <- E exp2(k sun_nd[l]) per layer, adds mu_sun sum E res to every level (E enters partial() with weight
// mu_sun / (2 pi), under the same non-finite rule).  The beam's row is the one four rows past the downward pass's first
// (row 8 of flux_rows): the pass reads S there and writes E at the surface over it, point by point, and the upward pass
// reads that row at each strip's start.  Lambertian (K3F_SUN): 1 - eps of it joins the diffuse term, S_i + mu_sun E / pi
// (added last, FP32).  Specular (K3F_SUN_SPECULAR): the reflected beam E_up = (1 - eps) E rises along mu_sun through
// the same layer factors and joins the level sums as above.  Where eps = 1, or E is not > 0 (an E of 0 times an FP32
// transmittance overflow next to 0 cm^-1 is NaN), nothing is reflected: a select, so the bits are those without the Sun.
constexpr int K3F_NO_SUN = 0, K3F_SUN = 1, K3F_SUN_SPECULAR = 2;

struct FluxLayer {
    float c2_over_t;         // 100 h c / kB / T_layer
    float nd[4];             // -depth log2(e) / mu_i: T_i = exp2(k * nd[i])
};

struct K3FSpan {
    int32_t seg0;            // the span's first segment
    int32_t nseg;            // how many segments it holds; -1: one, and the band covers all of the span's points
};

struct K3FArgs {
    float wmu[4];            // w_i mu_i
    float *rows;             // [NMU][ld_rows]: radiance leaving the column at the last level of the pass (NULL: none)
    int64_t ld_rows;
    double *part;            // [gridDim.x][n_layers + 1] per-CTA level sums; band pass: [n_layers + 1][ld_part]
    // band pass only
    const int32_t *strips;   // the n_list strips that meet a band, ascending
    int64_t n_list;
    const K3FSpan *spans;    // per span of the chunk, 8 per strip (a ragged last strip padded with empty spans)
    const uint32_t *seg_range;   // per segment: its points within the span, [lo, hi) as lo | hi << 16 (0 <= lo < hi <= 128)
    int64_t ld_part;         // the number of segments
    // boundaries only
    const float *eps;        // upward pass: the surface emissivity on the chunk
    const float *surf_down;  // upward pass: [NMU][ld_rows], the downward pass's radiance reaching the surface
    int32_t specular;        // upward pass: 1 specular reflection, 0 Lambertian
    float c2_over_ttop;      // downward pass: 100 h c / kB / T_top; 0: I = 0 at level L
    // solar beam only (K3FArgs stays within 128 bytes: a larger one changes the code of every instantiation)
    const float *sun_nd;     // [n_layers] -depth log2(e) / mu_sun: the beam's T = exp2(k * sun_nd[l])
    float sun_w;             // mu_sun / (2 pi): the beam's weight in partial() (the sums are scaled by 2 pi res)
    float sun_mu_over_pi;    // upward pass, Lambertian: mu_sun / pi, the diffuse radiance of a reflected unit beam
};
static_assert(sizeof(K3FArgs) <= 128, "K3FArgs above 128 bytes changes the compiled k3_flux_tma");

constexpr int K3F_WARPS = K3T_THREADS / 32;
struct K3FSmem {
    float k[K3T_SLOTS][K3T_LAYERS][K3T_STRIP];
    uint64_t full[K3T_SLOTS];
};                                                     // followed by double acc[K3F_WARPS][n_layers + 1]

// Resident CTAs per SM, from the register count without spills (-Xptxas -v, 256 threads): one and two nodes fit 64
// registers (4 CTAs; one node spills at the 48 of 5 CTAs), three and four nodes take 78-80 (3 CTAs).
__host__ __device__ constexpr int k3f_minb(int nmu) { return nmu <= 2 ? 4 : 3; }

__host__ __device__ constexpr size_t k3f_smem_bytes(int n_layers) {
    return sizeof(K3FSmem) + sizeof(double) * K3F_WARPS * (size_t)(n_layers + 1);
}

template <int NMU, bool DOWN, bool BAND = false, bool BOUND = false, int SUN = K3F_NO_SUN>
__global__ void __launch_bounds__(K3T_THREADS, k3f_minb(NMU))
k3_flux_tma(const float *__restrict__ kmat, int64_t ld, int n_layers, const FluxLayer *__restrict__ layers,
            int64_t n_chunk, int64_t i_begin, int64_t n_total, double x0, double dx, double x_last,
            float c2_over_tsurf, float nu_interp_min, const K3FArgs a) {
    static_assert(SUN == K3F_NO_SUN || BOUND, "the solar beam takes the boundary path");
    static_assert(!(DOWN && SUN == K3F_SUN_SPECULAR), "the downward beam does not depend on the reflection");
    constexpr bool BEAM = SUN != K3F_NO_SUN && (DOWN || SUN == K3F_SUN_SPECULAR);   // the pass carries a beam
    extern __shared__ __align__(128) unsigned char k3_smem_raw[];
    K3FSmem &sm = *reinterpret_cast<K3FSmem *>(k3_smem_raw);
    double *acc = reinterpret_cast<double *>(k3_smem_raw + sizeof(K3FSmem));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_levels = n_layers + 1;
    const int64_t n_strips = BAND ? a.n_list : (n_chunk + K3T_STRIP - 1) / K3T_STRIP;
    const int groups = (n_layers + K3T_LAYERS - 1) / K3T_LAYERS;
    const int64_t my_strips = blockIdx.x < n_strips ? (n_strips - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t n_steps = my_strips * groups;
    if constexpr (!BAND)
        for (int j = tid; j < K3F_WARPS * n_levels; j += K3T_THREADS) acc[j] = 0.0;
    if (tid == 0) {
        for (int s = 0; s < K3T_SLOTS; ++s) mbar_init(&sm.full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    // step s of the CTA covers row group s % groups of its strip, counted from the top for the downward pass
    auto group_of = [&](int64_t step) { const int g = (int)(step % groups); return DOWN ? groups - 1 - g : g; };
    auto strip_of = [&](int64_t step) {
        const int64_t s = blockIdx.x + (step / groups) * gridDim.x;
        return BAND ? (int64_t)a.strips[s] : s;
    };
    auto issue = [&](int64_t step) {                   // thread 0 only
        const int slot = (int)(step % K3T_SLOTS);
        const int64_t strip = strip_of(step);
        const int g = group_of(step);
        const int64_t p0 = strip * K3T_STRIP;
        const int64_t pts = min((int64_t)K3T_STRIP, ((n_chunk - p0) + 3) & ~int64_t(3));   // rows are padded to 4 floats
        const int rows = min(K3T_LAYERS, n_layers - g * K3T_LAYERS);
        mbar_expect_tx(&sm.full[slot], (uint32_t)(rows * pts * 4));
        for (int r = 0; r < rows; ++r)
            tma_bulk_g2s(sm.k[slot][r], kmat + (int64_t)(g * K3T_LAYERS + r) * ld + p0, (uint32_t)(pts * 4), &sm.full[slot]);
    };
    if (tid == 0)
        for (int64_t s = 0; s < min(n_steps, (int64_t)(K3T_SLOTS - 1)); ++s) issue(s);

    float nu[4], a3[4], rad[NMU][4];
    float beam[4] = {0.f, 0.f, 0.f, 0.f};              // BEAM: the solar beam at the thread's four points
    bool interp = false;
    int n_valid = 0;                                   // of the thread's four points, those inside the chunk
    int64_t i0 = 0;
    // sum_i w_i mu_i sum_q I_i(nu_q) over the thread's points inside the chunk.  A value that is not finite counts as 0:
    // the NaN of the 0 cm^-1 point, and the +-inf of the few points next to it where the reference's negative Doppler
    // widths make k < 0 and T = exp(-k u) overflows FP32.  The plain sum is checked once; the masked sum only runs for a
    // ragged last strip or when the plain sum met such a value.
    auto partial = [&]() {
        float s = 0.f;
        if (n_valid == 4) {
#pragma unroll
            for (int i = 0; i < NMU; ++i) {
                const float2 p = __fadd2_rn(make_float2(rad[i][0], rad[i][1]), make_float2(rad[i][2], rad[i][3]));
                s = fmaf(a.wmu[i], p.x + p.y, s);
            }
        }
        if (n_valid < 4 || !isfinite(s)) {
            s = 0.f;
#pragma unroll
            for (int i = 0; i < NMU; ++i) {
                float t = 0.f;
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (q < n_valid && isfinite(rad[i][q])) t += rad[i][q];
                s = fmaf(a.wmu[i], t, s);
            }
        }
        if constexpr (BEAM) {                          // + mu_sun / (2 pi) sum_q E(nu_q), the same non-finite rule
            float e = 0.f;
            if (n_valid == 4) {
                const float2 p = __fadd2_rn(make_float2(beam[0], beam[1]), make_float2(beam[2], beam[3]));
                e = p.x + p.y;
            }
            if (n_valid < 4 || !isfinite(e)) {
                e = 0.f;
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (q < n_valid && isfinite(beam[q])) e += beam[q];
            }
            s = fmaf(a.sun_w, e, s);
        }
        return s;
    };
    auto level_add = [&](float v, int level) {         // every lane of the warp takes part
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) acc[warp * n_levels + level] += (double)v;
    };
    // band pass: one value per segment of the warp's span.  A span inside one band takes partial() and the butterfly
    // above.  Otherwise each point's sum_i w_i mu_i I_i (a value that is not finite counts as 0) is formed once, and the
    // segments are taken two at a time: each a masked sum over the thread's points in its range [lo, hi) of the span,
    // both through one interleaved butterfly.
    auto band_add = [&](int level) {                   // every lane of the warp takes part; the span is the warp's
        const K3FSpan sp = a.spans[i0 >> 7];
        double *dst = a.part + (int64_t)level * a.ld_part + sp.seg0;
        if (sp.nseg < 0) {
            float v = partial();
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) dst[0] = (double)v;
        } else if (sp.nseg > 0) {
            float v[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                v[q] = 0.f;
#pragma unroll
                for (int i = 0; i < NMU; ++i)
                    if (isfinite(rad[i][q])) v[q] = fmaf(a.wmu[i], rad[i][q], v[q]);
                if constexpr (BEAM)
                    if (isfinite(beam[q])) v[q] = fmaf(a.sun_w, beam[q], v[q]);
            }
            for (int s = 0; s < sp.nseg; s += 2) {
                const uint32_t r0 = a.seg_range[sp.seg0 + s], r1 = s + 1 < sp.nseg ? a.seg_range[sp.seg0 + s + 1] : 0u;
                float t0 = 0.f, t1 = 0.f;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint32_t p = 4 * lane + q;
                    if (p >= (r0 & 0xffffu) && p < (r0 >> 16)) t0 += v[q];
                    if (p >= (r1 & 0xffffu) && p < (r1 >> 16)) t1 += v[q];
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    t0 += __shfl_xor_sync(0xffffffffu, t0, o);
                    t1 += __shfl_xor_sync(0xffffffffu, t1, o);
                }
                if (lane == 0) {
                    dst[s] = (double)t0;
                    if (s + 1 < sp.nseg) dst[s + 1] = (double)t1;
                }
            }
        }
    };
    auto add_level = [&](int level) {
        if constexpr (BAND) band_add(level);
        else level_add(partial(), level);
    };
    // v[q] = p[i0 + q] for the thread's points inside the chunk, 0 outside (solar beam only)
    auto chunk_load4 = [&](const float *p, float (&v)[4]) {
        if (n_valid == 4) {
            const float4 v4 = *reinterpret_cast<const float4 *>(p + i0);
            v[0] = v4.x; v[1] = v4.y; v[2] = v4.z; v[3] = v4.w;
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) v[q] = q < n_valid ? p[i0 + q] : 0.f;
        }
    };
    // boundaries, upward pass: rad holds B(nu, T_s); make it eps B + (1 - eps) S_i (points outside the chunk keep B)
    auto surface_start = [&]() {
        float eps[4] = {1.f, 1.f, 1.f, 1.f}, dn[NMU][4];
        if (n_valid == 4) {
            const float4 e4 = *reinterpret_cast<const float4 *>(a.eps + i0);
            eps[0] = e4.x; eps[1] = e4.y; eps[2] = e4.z; eps[3] = e4.w;
#pragma unroll
            for (int i = 0; i < NMU; ++i) {
                const float4 d4 = *reinterpret_cast<const float4 *>(a.surf_down + (int64_t)i * a.ld_rows + i0);
                dn[i][0] = d4.x; dn[i][1] = d4.y; dn[i][2] = d4.z; dn[i][3] = d4.w;
            }
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (q < n_valid) eps[q] = a.eps[i0 + q];
#pragma unroll
                for (int i = 0; i < NMU; ++i) dn[i][q] = q < n_valid ? a.surf_down[(int64_t)i * a.ld_rows + i0 + q] : 0.f;
            }
        }
        float es[4] = {0.f, 0.f, 0.f, 0.f};           // the solar beam reaching the surface
        if constexpr (SUN != K3F_NO_SUN) chunk_load4(a.surf_down + (int64_t)4 * a.ld_rows, es);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float s = 0.f;                             // Lambertian: F_down / pi = sum_j 2 w_j mu_j I_down_j
#pragma unroll
            for (int j = 0; j < NMU; ++j) s = fmaf(2.f * a.wmu[j], dn[j][q], s);
            if constexpr (SUN == K3F_SUN)              // + mu_sun E / pi
                if (es[q] > 0.f) s = fmaf(a.sun_mu_over_pi, es[q], s);
            if constexpr (SUN == K3F_SUN_SPECULAR)     // the reflected beam
                beam[q] = eps[q] == 1.f || !(es[q] > 0.f) ? 0.f : (1.f - eps[q]) * es[q];
#pragma unroll
            for (int i = 0; i < NMU; ++i) {
                const float sv = (SUN == K3F_NO_SUN ? a.specular != 0 : SUN == K3F_SUN_SPECULAR) ? dn[i][q] : s;
                rad[i][q] = eps[q] == 1.f ? rad[i][q] : fmaf(eps[q], rad[i][q], (1.f - eps[q]) * sv);
            }
        }
    };
    for (int64_t step = 0; step < n_steps; ++step) {
        const int slot = (int)(step % K3T_SLOTS);
        const int g = group_of(step);
        if (step % groups == 0) {                      // a new strip: the boundary radiance of the pass
            const int64_t strip = strip_of(step);
            if constexpr (SUN != K3F_NO_SUN) {          // (read again: 4 tid held over the strips would spill)
                uint32_t t;
                asm volatile("mov.u32 %0, %%tid.x;" : "=r"(t));
                i0 = strip * K3T_STRIP + 4 * (int)t;
            } else {
                i0 = strip * K3T_STRIP + 4 * tid;
            }
            n_valid = (int)max((int64_t)0, min((int64_t)4, n_chunk - i0));
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double x = axis_value(i_begin + i0 + q, n_total, x0, dx, x_last);
                nu[q] = (float)x;
                a3[q] = (float)(2E8 * hPlanck * (cLight * cLight) * (x * x * x));
                float r0 = DOWN ? 0.f : planck_f32(a3[q], c2_over_tsurf * nu[q]);
                if constexpr (BOUND && DOWN)
                    if (a.c2_over_ttop > 0.f) r0 = planck_f32(a3[q], a.c2_over_ttop * nu[q]);   // B(nu, T_top)
#pragma unroll
                for (int i = 0; i < NMU; ++i) rad[i][q] = r0;
            }
            if constexpr (BOUND && !DOWN) surface_start();
            if constexpr (BEAM && DOWN) chunk_load4(a.rows + (int64_t)4 * a.ld_rows, beam);   // E = S(nu) at level L
            interp = nu[0] >= nu_interp_min;
            if (!DOWN) add_level(0);                   // (the plain downward pass starts from 0 at level L,
            else if (BAND || BOUND) add_level(n_layers);   // whose band segment slots must still be written: zeros)
        }
        if (tid == 0 && step + K3T_SLOTS - 1 < n_steps) issue(step + K3T_SLOTS - 1);
        mbar_wait(&sm.full[slot], (uint32_t)((step / K3T_SLOTS) & 1));
        const int rows = min(K3T_LAYERS, n_layers - g * K3T_LAYERS);
#pragma unroll
        for (int rr = 0; rr < K3T_LAYERS; ++rr) {
            if (rr < rows) {
                const int r = DOWN ? rows - 1 - rr : rr;
                const int l = g * K3T_LAYERS + r;
                const float4 k4 = *reinterpret_cast<const float4 *>(&sm.k[slot][r][4 * tid]);
                const FluxLayer fl = layers[l];
                float b[4];
                k3_planck4(nu, a3, fl.c2_over_t, interp, b);
                const float2 b01 = make_float2(b[0], b[1]), b23 = make_float2(b[2], b[3]);
#pragma unroll
                for (int i = 0; i < NMU; ++i) {
                    const float2 nd = make_float2(fl.nd[i], fl.nd[i]);
                    const float2 e01 = __fmul2_rn(make_float2(k4.x, k4.y), nd), e23 = __fmul2_rn(make_float2(k4.z, k4.w), nd);
                    const float2 r01 = k3_fold_step2(make_float2(rad[i][0], rad[i][1]), e01, b01);
                    const float2 r23 = k3_fold_step2(make_float2(rad[i][2], rad[i][3]), e23, b23);
                    rad[i][0] = r01.x; rad[i][1] = r01.y; rad[i][2] = r23.x; rad[i][3] = r23.y;
                }
                if constexpr (BEAM) {                  // E <- E exp(-k depth / mu_sun): no emission, no scattering
                    const float2 nd = make_float2(a.sun_nd[l], a.sun_nd[l]);
                    const float2 e01 = __fmul2_rn(make_float2(k4.x, k4.y), nd), e23 = __fmul2_rn(make_float2(k4.z, k4.w), nd);
                    const float2 t01 = make_float2(k3_ex2(e01.x), k3_ex2(e01.y)), t23 = make_float2(k3_ex2(e23.x), k3_ex2(e23.y));
                    const float2 b01 = __fmul2_rn(make_float2(beam[0], beam[1]), t01);
                    const float2 b23 = __fmul2_rn(make_float2(beam[2], beam[3]), t23);
                    beam[0] = b01.x; beam[1] = b01.y; beam[2] = b23.x; beam[3] = b23.y;
                }
                add_level(DOWN ? l : l + 1);
            }
        }
        __syncthreads();                               // every thread is done with this slot: it may be refilled
        if (step % groups == groups - 1 && a.rows && n_valid > 0) {
#pragma unroll
            for (int i = 0; i < NMU; ++i) {
                float *dst = a.rows + (int64_t)i * a.ld_rows + i0;
                if (n_valid == 4) *reinterpret_cast<float4 *>(dst) = make_float4(rad[i][0], rad[i][1], rad[i][2], rad[i][3]);
                else
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        if (q < n_valid) dst[q] = rad[i][q];
            }
        }
        if constexpr (BEAM && DOWN) {                  // the beam at the surface, for the upward pass
            if (step % groups == groups - 1 && n_valid > 0) {
                float *dst = a.rows + (int64_t)4 * a.ld_rows + i0;
                if (n_valid == 4) *reinterpret_cast<float4 *>(dst) = make_float4(beam[0], beam[1], beam[2], beam[3]);
                else
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        if (q < n_valid) dst[q] = beam[q];
            }
        }
    }
    if constexpr (!BAND) {
        __syncthreads();
        for (int j = tid; j < n_levels; j += K3T_THREADS) {
            double s = 0.0;
            for (int w = 0; w < K3F_WARPS; ++w) s += acc[w * n_levels + j];
            a.part[(int64_t)blockIdx.x * n_levels + j] = s;
        }
    }
}

// Surface emissivity of the boundaries on the owned chunk: eps[i] = np.interp(x, table_nu, table_eps) in FP64 (numpy's
// arithmetic), rounded to FP32; x the Planck axis of the fold.  tab = table_nu | table_eps, n_tab entries each.
__global__ void __launch_bounds__(256)
k3_flux_emissivity(int64_t n_chunk, int64_t i_begin, int64_t n_total, double x0, double dx, double x_last,
                   const double *__restrict__ tab, int64_t n_tab, float *__restrict__ eps) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_chunk; i += (int64_t)gridDim.x * blockDim.x)
        eps[i] = (float)np_interp(axis_value(i_begin + i, n_total, x0, dx, x_last), tab, tab + n_tab, n_tab);
}

// Solar irradiance at the top on the owned chunk: s[i] = np.interp(x, table_nu, table_s, left=0, right=0) in FP64,
// rounded to FP32; x the Planck axis of the fold.  tab = table_nu | table_s, n_tab >= 2 entries each.
__global__ void __launch_bounds__(256)
k3_flux_solar(int64_t n_chunk, int64_t i_begin, int64_t n_total, double x0, double dx, double x_last,
              const double *__restrict__ tab, int64_t n_tab, float *__restrict__ s) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_chunk; i += (int64_t)gridDim.x * blockDim.x) {
        const double x = axis_value(i_begin + i, n_total, x0, dx, x_last);
        s[i] = x < tab[0] || x > tab[n_tab - 1] ? 0.f : (float)np_interp(x, tab, tab + n_tab, n_tab);
    }
}

// ---- water-vapour continuum (prb_set_continuum), added to the k matrix before the fold -----------------------------
//   k_c,l(nu) = n_l rho_l R(nu, T_l) [x_l (t_ref/T_l)^n(nu) C_s(nu) + (1 - x_l) C_f(nu)]
//   n_l = x_l P_l / 1e4 / kB / T_l,  rho_l = (P_l / p_ref)(t_ref / T_l),  R(nu, T) = nu tanh(c2 nu / 2T)
// in MT_CKD's form.  MT_CKD's coefficients are defined against lines cut at 25 cm^-1 with the 25 cm^-1 value subtracted;
// this path cuts at 5 P/p0 cm^-1 and adds whatever table it is given: matching the two is the caller's job.

// The table on the owned chunk, once per (grid, table): rows [0, ld) C_s, [ld, 2 ld) C_f, [2 ld, 3 ld) n, each
// np.interp in FP64 (numpy's arithmetic) rounded to FP32; C_s and C_f are 0 outside the table, n is clamped there.  Points
// from n_chunk up to ld (the row padding) get 0 in all three.  tab = table_nu | c_self | c_foreign | t_exp, n_tab each.
__global__ void __launch_bounds__(256)
k3_continuum_rows(int64_t n_chunk, int64_t ld, int64_t i_begin, int64_t n_total, double x0, double dx, double x_last,
                  const double *__restrict__ tab, int64_t n_tab, float *__restrict__ rows) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ld; i += (int64_t)gridDim.x * blockDim.x) {
        float cs = 0.f, cf = 0.f, n = 0.f;
        if (i < n_chunk) {
            const double x = axis_value(i_begin + i, n_total, x0, dx, x_last);
            const bool inside = !(x < tab[0] || x > tab[n_tab - 1]);
            cs = inside ? (float)np_interp(x, tab, tab + n_tab, n_tab) : 0.f;
            cf = inside ? (float)np_interp(x, tab, tab + 2 * n_tab, n_tab) : 0.f;
            n = (float)np_interp(x, tab, tab + 3 * n_tab, n_tab);
        }
        rows[i] = cs;
        rows[ld + i] = cf;
        rows[2 * ld + i] = n;
    }
}

// A layer of the add, formed on the host in FP64 and rounded once: the products n rho x and n rho (1 - x) never leave
// the normal FP32 range, where x C_s alone (1e-6 x 1e-30 in the stratosphere) would reach the flush-to-zero range.
struct ContLayer {
    float a;                 // n_l rho_l x_l
    float b;                 // n_l rho_l (1 - x_l)
    float log2_tref_t;       // log2(t_ref / T_l)
    float c2_over_2t;        // c2 / (2 T_l)
    int row;                 // the layer's row of the k matrix
    int pad;
};

// tanh(y) for y >= 0, to a few FP32 ulp relative everywhere: next to 0 cm^-1, y = c2 nu / 2T is ~3e-6, where
// (1 - e^-2y) / (1 + e^-2y) would lose every digit to cancellation.  Below 1/4 the odd series to y^9 (truncation < 1e-8
// relative), above it that quotient with e^-2y <= 0.61 (one ex2, one rcp).
__device__ __forceinline__ float k3_cont_tanh(float y) {
    if (y < 0.25f) {
        const float y2 = y * y;
        float p = fmaf(y2, 2.1869488536e-2f, -5.3968253968e-2f);      // 62/2835, -17/315
        p = fmaf(y2, p, 1.3333333333e-1f);                             // 2/15
        p = fmaf(y2, p, -3.3333333333e-1f);                            // -1/3
        return fmaf(y * y2, p, y);
    }
    const float t = k3_ex2(y * -2.8853900817779268f);                // e^-2y
    return (1.f - t) * k3_rcp(1.f + t);
}

// k[row][i] += k_c(nu_i) for the listed layers (those with x_l > 0; no other row is read or written), on the owned chunk.
// A thread owns four points (one float4: ld is a multiple of 4), loads their C_s, C_f, n once and walks the layers,
// K3_CONT_UNROLL rows' loads in flight before their math.  A pointwise function of the chunk: no atomics, and
// tile-aligned chunks give the rows of the whole grid bit for bit.
constexpr int K3_CONT_UNROLL = 4;
__global__ void __launch_bounds__(256)
k3_continuum_add(float *__restrict__ kmat, int64_t ld, const ContLayer *__restrict__ layers, int n_list,
                 const float *__restrict__ rows, int64_t i_begin, int64_t n_total, double x0, double dx, double x_last) {
    const int64_t nvec = ld >> 2;
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i0 = v << 2;
        const float4 cs4 = *reinterpret_cast<const float4 *>(rows + i0);
        const float4 cf4 = *reinterpret_cast<const float4 *>(rows + ld + i0);
        const float4 n4 = *reinterpret_cast<const float4 *>(rows + 2 * ld + i0);
        const float cs[4] = {cs4.x, cs4.y, cs4.z, cs4.w}, cf[4] = {cf4.x, cf4.y, cf4.z, cf4.w};
        const float nn[4] = {n4.x, n4.y, n4.z, n4.w};
        float nu[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) nu[q] = (float)axis_value(i_begin + i0 + q, n_total, x0, dx, x_last);
        for (int j0 = 0; j0 < n_list; j0 += K3_CONT_UNROLL) {
            float4 k4[K3_CONT_UNROLL];
#pragma unroll
            for (int j = 0; j < K3_CONT_UNROLL; ++j)
                if (j0 + j < n_list) k4[j] = *reinterpret_cast<const float4 *>(kmat + (int64_t)layers[j0 + j].row * ld + i0);
#pragma unroll
            for (int j = 0; j < K3_CONT_UNROLL; ++j) {
                if (j0 + j < n_list) {
                    const ContLayer c = layers[j0 + j];
                    float kk[4] = {k4[j].x, k4[j].y, k4[j].z, k4[j].w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        // (t_ref/T)^n as one ex2; the clamp keeps it finite, so a zero coefficient gives exactly 0
                        const float tn = k3_ex2(fminf(nn[q] * c.log2_tref_t, 126.f));
                        const float r = nu[q] * k3_cont_tanh(c.c2_over_2t * nu[q]);
                        kk[q] += r * fmaf(c.a, tn * cs[q], c.b * cf[q]);
                    }
                    *reinterpret_cast<float4 *>(kmat + (int64_t)c.row * ld + i0) = make_float4(kk[0], kk[1], kk[2], kk[3]);
                }
            }
        }
    }
}

// Band totals of the band pass: out[d][b][j] = scale * sum of band b's segments at level j of pass d (0 up, 1 down), for
// the bands list[0 .. n_list).  G threads take one (d, b, j): thread t adds segments t, t + G, ... in order, then a fixed
// xor butterfly over the warp and, for G = 256, the eight warps' values in a fixed tree.  The host picks G from the
// band's segment count only (256 above K3F_BAND_WARP_MAX segments, else 32), so the order is a function of that count.
constexpr int K3F_BAND_WARP_MAX = 1024;
template <int G>
__global__ void __launch_bounds__(256)
k3_flux_band_sum(const double *__restrict__ part, int64_t ld_part, int n_levels, const int32_t *__restrict__ list,
                 int n_list, const int32_t *__restrict__ band_seg, int n_bands, double scale, double *__restrict__ out) {
    constexpr int PER = 256 / G;                       // (d, b, j) per block
    const int64_t item = (int64_t)blockIdx.x * PER + threadIdx.x / G;
    if (item >= 2 * (int64_t)n_list * n_levels) return;    // uniform over each group of G threads
    const int t = threadIdx.x % G, lane = threadIdx.x & 31;
    const int j = (int)(item % n_levels);
    const int64_t r = item / n_levels;
    const int d = (int)(r / n_list), b = list[r % n_list];
    const int32_t s0 = band_seg[b], cnt = band_seg[b + 1] - s0;
    const double *p = part + ((int64_t)d * n_levels + j) * ld_part + s0;
    double s = 0.0;
    for (int k = t; k < cnt; k += G) s += p[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if constexpr (G == 256) {
        __shared__ double w[8];
        if (lane == 0) w[threadIdx.x >> 5] = s;
        __syncthreads();
        s = ((w[0] + w[1]) + (w[2] + w[3])) + ((w[4] + w[5]) + (w[6] + w[7]));
    }
    if (t == 0) out[((int64_t)d * n_bands + b) * n_levels + j] = s * scale;
}

// out[j] = scale * sum over the n_parts CTAs, in CTA order, of their level-j partials.
__global__ void __launch_bounds__(256)
k3_flux_sum(const double *__restrict__ part, int n_parts, int n_levels, double scale, double *__restrict__ out) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n_levels; j += gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int b = 0; b < n_parts; ++b) s += part[(int64_t)b * n_levels + j];
        out[j] = s * scale;
    }
}

// ---- layer kernels: the change of the outgoing and surface fluxes when one layer's state is swapped ------------------
// prb_atmosphere_save_base keeps a copy of the column (the base) and its FP64 optical depth S = sum_l k_l d_l per point;
// prb_atmosphere_layer_kernels compares it with the current column layer by layer.  With T_l = exp(-k_l d_l / mu) and the
// primed values those of the current column, swapping layer l alone changes the radiance leaving it by
//   up:   dI_{l+1} = (1 - T'_l)(B'_l - B_l) + (T'_l - T_l)(I_l - B_l)        I_l the base radiance entering from below
//   down: dI_l     = (1 - T'_l)(B'_l - B_l) + (T'_l - T_l)(I_{l+1} - B_l)    I_{l+1} the base radiance entering from above
// and the fold is linear in what enters, so that change reaches the top (the surface) multiplied by the base
// transmittance of the layers above (below): exp(-rem / mu), rem = S minus the depths of layer l and those before it in
// the pass's order, formed in FP64 by subtracting k_l d_l from S layer by layer (rem is small exactly where the kernels
// live, the top layers of an opaque band, while S itself may be 1e6).  Both differences are formed without cancellation:
//   T'_l - T_l = T_l (2^de - 1) for small de, else T'_l - T_l directly (k3_dtrans); de = k' nd' - k nd is formed as
//   (k' - k) nd + k' (nd' - nd), nd' - nd on the host in FP64, so neither a row change nor a depth change cancels (and
//   de = 0 exactly for equal rows and depths);
//   B'_l - B_l = B_l (e^(x - x') - 1) / (1 - e^-x'), x = c2 nu / T, x - x' formed on the host in FP64 (exactly 0 for
//   equal temperatures).
// So a layer whose row, depth and temperature are bit-identical in both columns adds exactly 0.  B_l follows the base
// column's Planck policy (k3_planck4 above its nu_interp_min), and B'_l - B_l is interpolated the same way.  The upward
// pass adds the surface entry exp(-S / mu)(B(T'_s) - B(T_s)) at level 0; the downward pass writes 0 there.  Sums as the
// band pass: per point sum_i w_i mu_i (...) (a term that is not finite counts as 0), per segment of the warp's span an
// FP32 butterfly and one FP64 store, then k3_flux_band_sum over "levels" 0..L.  No atomics.
constexpr int K3K_LAYERS = 2;                          // layers per ring slot: two rows each (base, current), 16 KB
constexpr int K3K_SLOTS = 2;

struct KernLayer {
    double depth;            // base depth_l (cm), for rem
    float c2_over_t;         // base 100 h c / kB / T_l
    float dx2;               // (c2 / T_l - c2 / T'_l) log2(e): x - x' in log2 units per cm-1
    float x2_cur;            // c2 / T'_l log2(e)
    float pad;
    float nd[4];             // base -depth_l log2(e) / mu_i
    float dnd[4];            // -(depth'_l - depth_l) log2(e) / mu_i, formed in FP64 (exactly 0 for equal depths)
};

struct K3KArgs {
    const float *base;       // [n_layers][ld] the base k matrix
    const double *s;         // [ld] the base optical depth
    const KernLayer *layers;
    float wmu[4];            // w_i mu_i
    float cu[4];             // -log2(e) / mu_i: exp(-rem / mu_i) = 2^(rem cu[i])
    float c2_over_ttop;      // downward pass: 100 h c / kB / T_top; 0: I = 0 at level L
    float c2_over_ts;        // upward pass, the surface: base 100 h c / kB / T_s
    float ts_dx2, ts_x2_cur; // ... and its dx2, x2_cur as KernLayer's
    double *part;            // [n_levels][ld_part] per-segment sums of the pass
    const int32_t *strips;   // the n_list strips that meet a band, ascending
    int64_t n_list;
    const K3FSpan *spans;    // as K3FArgs
    const uint32_t *seg_range;
    int64_t ld_part;
};

struct K3KSmem {
    float k[K3K_SLOTS][K3K_LAYERS][2][K3T_STRIP];
    uint64_t full[K3K_SLOTS];
};

// Resident CTAs per SM the registers allow without spills (-Xptxas -v, 256 threads): one node fits 80 registers
// (3 CTAs), two to four take 116-123 (2 CTAs; two nodes spill at 80).
__host__ __device__ constexpr int k3k_minb(int nmu) { return nmu == 1 ? 3 : 2; }

// 2^e - 1 to a few FP32 ulp relative: the fold's five-term series below |e| = 1/8 (exactly 0 at e = 0), else ex2 - 1.
__device__ __forceinline__ float k3_exp2m1(float e) {
    float p = fmaf(e, 1.3333558146e-3f, 9.6181291076e-3f);
    p = fmaf(e, p, 5.5504108665e-2f);
    p = fmaf(e, p, 2.4022650696e-1f);
    p = fmaf(e, p, 6.9314718056e-1f);
    return fabsf(e) < 0.125f ? e * p : k3_ex2(e) - 1.0f;
}

// T' - T = 2^(e + de) - 2^e: 2^e (2^de - 1) by the series below |de| = 1/8 (exactly 0 at de = 0), else the plain
// difference, which cancels little there and stays finite where 2^e underflows and 2^de overflows (an opaque layer).
__device__ __forceinline__ float k3_dtrans(float e, float de) {
    float p = fmaf(de, 1.3333558146e-3f, 9.6181291076e-3f);
    p = fmaf(de, p, 5.5504108665e-2f);
    p = fmaf(de, p, 2.4022650696e-1f);
    p = fmaf(de, p, 6.9314718056e-1f);
    return fabsf(de) < 0.125f ? k3_ex2(e) * (de * p) : k3_ex2(e + de) - k3_ex2(e);
}

// B(T') - B(T) from b = B(T): b (e^(x - x') - 1) / (1 - e^-x'), with dx2 = (x - x') log2(e), x2c = x' log2(e).
__device__ __forceinline__ float k3_dplanck(float b, float x2c, float dx2) {
    return b * k3_exp2m1(dx2) / -k3_exp2m1(-x2c);
}

template <int NMU, bool DOWN>
__global__ void __launch_bounds__(K3T_THREADS, k3k_minb(NMU))
k3_kernel_tma(const float *__restrict__ kmat, int64_t ld, int n_layers, int64_t n_chunk, int64_t i_begin, int64_t n_total,
              double x0, double dx, double x_last, float nu_interp_min, const K3KArgs a) {
    extern __shared__ __align__(128) unsigned char k3_smem_raw[];
    K3KSmem &sm = *reinterpret_cast<K3KSmem *>(k3_smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    const int groups = (n_layers + K3K_LAYERS - 1) / K3K_LAYERS;
    const int64_t my_strips = blockIdx.x < a.n_list ? (a.n_list - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t n_steps = my_strips * groups;
    if (tid == 0) {
        for (int s = 0; s < K3K_SLOTS; ++s) mbar_init(&sm.full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    auto group_of = [&](int64_t step) { const int g = (int)(step % groups); return DOWN ? groups - 1 - g : g; };
    auto strip_of = [&](int64_t step) { return (int64_t)a.strips[blockIdx.x + (step / groups) * gridDim.x]; };
    auto issue = [&](int64_t step) {                   // thread 0 only: both rows of every layer of the group
        const int slot = (int)(step % K3K_SLOTS);
        const int g = group_of(step);
        const int64_t p0 = strip_of(step) * K3T_STRIP;
        const int64_t pts = min((int64_t)K3T_STRIP, ((n_chunk - p0) + 3) & ~int64_t(3));
        const int rows = min(K3K_LAYERS, n_layers - g * K3K_LAYERS);
        mbar_expect_tx(&sm.full[slot], (uint32_t)(2 * rows * pts * 4));
        for (int r = 0; r < rows; ++r) {
            const int64_t off = (int64_t)(g * K3K_LAYERS + r) * ld + p0;
            tma_bulk_g2s(sm.k[slot][r][0], a.base + off, (uint32_t)(pts * 4), &sm.full[slot]);
            tma_bulk_g2s(sm.k[slot][r][1], kmat + off, (uint32_t)(pts * 4), &sm.full[slot]);
        }
    };
    if (tid == 0)
        for (int64_t s = 0; s < min(n_steps, (int64_t)(K3K_SLOTS - 1)); ++s) issue(s);

    float nu[4], a3[4], rad[NMU][4];
    double rem[4];
    bool interp = false;
    int n_valid = 0;
    int64_t i0 = 0;
    // the per-point values v of one level into its segments: a masked FP32 sum per segment, an xor butterfly, one FP64
    // store by lane 0 (points outside the chunk hold v = 0)
    auto seg_add = [&](const float (&v)[4], int level) {
        const K3FSpan sp = a.spans[i0 >> 7];
        if (sp.nseg == 0) return;
        const int nseg = sp.nseg < 0 ? 1 : sp.nseg;
        double *dst = a.part + (int64_t)level * a.ld_part + sp.seg0;
        for (int s = 0; s < nseg; s += 2) {
            const uint32_t r0 = sp.nseg < 0 ? 128u << 16 : a.seg_range[sp.seg0 + s];
            const uint32_t r1 = s + 1 < nseg ? a.seg_range[sp.seg0 + s + 1] : 0u;
            float t0 = 0.f, t1 = 0.f;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t p = 4 * lane + q;
                if (p >= (r0 & 0xffffu) && p < (r0 >> 16)) t0 += v[q];
                if (p >= (r1 & 0xffffu) && p < (r1 >> 16)) t1 += v[q];
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                t0 += __shfl_xor_sync(0xffffffffu, t0, o);
                t1 += __shfl_xor_sync(0xffffffffu, t1, o);
            }
            if (lane == 0) {
                dst[s] = (double)t0;
                if (s + 1 < nseg) dst[s + 1] = (double)t1;
            }
        }
    };
    for (int64_t step = 0; step < n_steps; ++step) {
        const int slot = (int)(step % K3K_SLOTS);
        const int g = group_of(step);
        if (step % groups == 0) {                      // a new strip: the boundary radiance of the pass, rem = S
            i0 = strip_of(step) * K3T_STRIP + 4 * tid;
            n_valid = (int)max((int64_t)0, min((int64_t)4, n_chunk - i0));
            float v[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double x = axis_value(i_begin + i0 + q, n_total, x0, dx, x_last);
                nu[q] = (float)x;
                a3[q] = (float)(2E8 * hPlanck * (cLight * cLight) * (x * x * x));
                rem[q] = q < n_valid ? a.s[i0 + q] : 0.0;
                float r0 = 0.f;
                if (!DOWN) r0 = planck_f32(a3[q], a.c2_over_ts * nu[q]);
                else if (a.c2_over_ttop > 0.f) r0 = planck_f32(a3[q], a.c2_over_ttop * nu[q]);
#pragma unroll
                for (int i = 0; i < NMU; ++i) rad[i][q] = r0;
                v[q] = 0.f;
                if (!DOWN && q < n_valid) {            // the surface entry: exp(-S / mu_i) (B(T'_s) - B(T_s))
                    const float db = k3_dplanck(r0, a.ts_x2_cur * nu[q], a.ts_dx2 * nu[q]);
                    const float rf = (float)rem[q];
#pragma unroll
                    for (int i = 0; i < NMU; ++i) {
                        const float c = k3_ex2(rf * a.cu[i]) * db;
                        if (isfinite(c)) v[q] = fmaf(a.wmu[i], c, v[q]);
                    }
                }
            }
            interp = nu[0] >= nu_interp_min;
            seg_add(v, 0);
        }
        if (tid == 0 && step + K3K_SLOTS - 1 < n_steps) issue(step + K3K_SLOTS - 1);
        mbar_wait(&sm.full[slot], (uint32_t)((step / K3K_SLOTS) & 1));
        const int rows = min(K3K_LAYERS, n_layers - g * K3K_LAYERS);
#pragma unroll
        for (int rr = 0; rr < K3K_LAYERS; ++rr) {
            if (rr < rows) {
                const int r = DOWN ? rows - 1 - rr : rr;
                const int l = g * K3K_LAYERS + r;
                // the rows are read from shared memory again for every node: held in registers they spill
                const float4 *kb4 = reinterpret_cast<const float4 *>(&sm.k[slot][r][0][4 * tid]);
                const float4 *kc4 = reinterpret_cast<const float4 *>(&sm.k[slot][r][1][4 * tid]);
                const KernLayer &fl = a.layers[l];
                float b[4], db[4], v[4];
                k3_planck4(nu, a3, fl.c2_over_t, interp, b);
                if (interp) {                          // B' - B at the first and last point, linear between
                    const float da = k3_dplanck(b[0], fl.x2_cur * nu[0], fl.dx2 * nu[0]);
                    const float dd = k3_dplanck(b[3], fl.x2_cur * nu[3], fl.dx2 * nu[3]);
                    const float d = dd - da;
                    db[0] = da; db[1] = fmaf(d, 1.0f / 3.0f, da); db[2] = fmaf(d, 2.0f / 3.0f, da); db[3] = dd;
                } else {
#pragma unroll
                    for (int q = 0; q < 4; ++q) db[q] = k3_dplanck(b[q], fl.x2_cur * nu[q], fl.dx2 * nu[q]);
                }
                {
                    const float4 k4 = *kb4;
                    const double d = fl.depth;
                    rem[0] = fma(-(double)k4.x, d, rem[0]); rem[1] = fma(-(double)k4.y, d, rem[1]);
                    rem[2] = fma(-(double)k4.z, d, rem[2]); rem[3] = fma(-(double)k4.w, d, rem[3]);
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) v[q] = 0.f;
#pragma unroll
                for (int i = 0; i < NMU; ++i) {
                    const float4 kb4i = *kb4, kc4i = *kc4;
                    const float kb[4] = {kb4i.x, kb4i.y, kb4i.z, kb4i.w}, kc[4] = {kc4i.x, kc4i.y, kc4i.z, kc4i.w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float e = kb[q] * fl.nd[i];
                        const float de = fmaf(kc[q] - kb[q], fl.nd[i], kc[q] * fl.dnd[i]);  // k' nd' - k nd
                        const float dt = k3_dtrans(e, de);                                  // T' - T
                        const float di = fmaf(-k3_exp2m1(e + de), db[q], dt * (rad[i][q] - b[q]));
                        const float c = k3_ex2((float)rem[q] * a.cu[i]) * di;
                        if (q < n_valid && isfinite(c)) v[q] = fmaf(a.wmu[i], c, v[q]);
                    }
                    const float2 nd = make_float2(fl.nd[i], fl.nd[i]);
                    const float2 e01 = __fmul2_rn(make_float2(kb[0], kb[1]), nd), e23 = __fmul2_rn(make_float2(kb[2], kb[3]), nd);
                    const float2 r01 = k3_fold_step2(make_float2(rad[i][0], rad[i][1]), e01, make_float2(b[0], b[1]));
                    const float2 r23 = k3_fold_step2(make_float2(rad[i][2], rad[i][3]), e23, make_float2(b[2], b[3]));
                    rad[i][0] = r01.x; rad[i][1] = r01.y; rad[i][2] = r23.x; rad[i][3] = r23.y;
                }
                seg_add(v, l + 1);
            }
        }
        __syncthreads();                               // every thread is done with this slot: it may be refilled
    }
}

// The base of the layer kernels: base = kmat row by row (streaming), and s[i] = sum_l k_l(i) depth_l in FP64, layer
// order, over all ld points of a row (the padding too, so the kernel passes may read any point of a float4).
__global__ void __launch_bounds__(256)
k3_kernel_base(const float *__restrict__ kmat, float *__restrict__ base, int64_t ld, int n_layers,
               const double *__restrict__ depth, double *__restrict__ s) {
    const int64_t nvec = ld >> 2;
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i0 = v << 2;
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
        for (int l0 = 0; l0 < n_layers; l0 += K3_UNROLL) {
            float4 k4[K3_UNROLL];
#pragma unroll
            for (int j = 0; j < K3_UNROLL; ++j)
                if (l0 + j < n_layers) k4[j] = __ldcs(reinterpret_cast<const float4 *>(kmat + (int64_t)(l0 + j) * ld + i0));
#pragma unroll
            for (int j = 0; j < K3_UNROLL; ++j) {
                if (l0 + j < n_layers) {
                    __stcs(reinterpret_cast<float4 *>(base + (int64_t)(l0 + j) * ld + i0), k4[j]);
                    const double d = depth[l0 + j];
                    acc[0] = fma((double)k4[j].x, d, acc[0]);
                    acc[1] = fma((double)k4[j].y, d, acc[1]);
                    acc[2] = fma((double)k4[j].z, d, acc[2]);
                    acc[3] = fma((double)k4[j].w, d, acc[3]);
                }
            }
        }
        *reinterpret_cast<double2 *>(s + i0) = make_double2(acc[0], acc[1]);
        *reinterpret_cast<double2 *>(s + i0 + 2) = make_double2(acc[2], acc[3]);
    }
}

// ---- cross-GPU completion barrier of one gather step ------------------------------------------------
// Launched (one warp) after the kernel that stored this rank's spectra into every peer's gather buffer.
// Lane p publishes "rank r finished epoch E" into peer p's flag block with a system-scope release, then
// waits until peer p's flag for E has arrived here: when the kernel retires, every rank's slot of the LOCAL
// gather buffer is complete.  A peer that never arrives trips the timeout and sets *err (reported by the host
// as PRB_ERR_PEER) instead of hanging the GPU.
struct PeerSignal {
    unsigned int *flags[K3_MAX_PEERS]; // every rank's flag block (own one included), [2][K3_MAX_PEERS] words each
    int rank, world;
    unsigned int epoch;
    unsigned int *err;
    unsigned long long timeout_ns;
};

__global__ void k_peer_signal_wait(const PeerSignal s) {
    const int p = threadIdx.x;
    if (p >= s.world) return;
    const int par = s.epoch & 1u;
    __threadfence_system();
    unsigned int *remote = s.flags[p] + par * K3_MAX_PEERS + s.rank;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(remote), "r"(s.epoch) : "memory");
    const unsigned int *mine = s.flags[s.rank] + par * K3_MAX_PEERS + p;
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (true) {
        unsigned int v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
        if ((int)(v - s.epoch) >= 0) break;
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > s.timeout_ns) { atomicOr(s.err, 1u); break; }
        __nanosleep(200);
    }
}

}  // namespace prb
