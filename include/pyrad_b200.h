/* pyrad_b200.h -- C ABI of libpyrad_b200.so, the B200 (sm_100a) engine behind PyRad's
 * gas-cell / atmosphere line-by-line path.
 *
 * The reference (bschrag620/PyRad) is pure Python + numpy and has NO plugin / FFI
 * interface (SURVEY.md section 8(b)).  The seam this library replaces is the method
 * edge between the host object model and the numpy physics:
 *
 *   pyradClasses.py:361-407  Isotope.createCrossSection   -> prb_upload_lines + prb_set_grid
 *                                                            + prb_layer_prepass + prb_line_sum
 *   pyradClasses.py:252-263  Line.broadenedLine/lorentzHW/gaussianHW      \
 *   pyradIntensity.py:16-32  intensityFactor                               > prb_layer_prepass (K1)
 *   pyradLineshape.py:22-29,58-71 half widths, pseudo-Voigt f and eta      /
 *   pyradLineshape.py:32-76  gaussian/lorentz/pseudoVoigt shapes + the scatter loop
 *                            pyradClasses.py:392-400                       -> prb_line_sum (K2)
 *   pyradClasses.py:581-587,707-716 absCoef / transmittance                \
 *   pyradPlanck.py:38-44     planckWavenumber                               > prb_layer_stream (K3)
 *   pyradClasses.py:784-787  Layer.transmission                            /
 *   pyradClasses.py:159-162,493-500 xsc np.interp + aligned placement      -> prb_xsc_place
 *   pyradUtilities.py:515-597 changeResXscFile / mergeXsc (file re-gridding) -> prb_parse_xsc_text + prb_xsc_place
 *   pyradUtilities.py:173-189,421-448 HITRAN-online CSV rows -> line arrays -> prb_ingest_hitran_csv
 *   pyradClasses.py:409-428,26-29 line survey, integrateSpectrum            -> prb_line_survey, prb_integrate_spectrum
 *   (absent upstream, SURVEY 3.5) multi-layer fold of Layer.transmission   -> prb_atmosphere
 *   (absent upstream) hemispheric fluxes, downwelling and slant radiances of the column -> prb_atmosphere_fluxes
 *   (absent upstream) the column's fluxes per wavenumber band, at every level      -> prb_atmosphere_band_fluxes
 *   (absent upstream) a grey or spectral surface and a warm top for both flux calls -> prb_set_flux_boundaries
 *   (absent upstream) an absorbed, reflected solar beam for both flux calls        -> prb_set_solar_source
 *   (absent upstream) a water-vapour continuum in the column's k matrix            -> prb_set_continuum
 *
 * Conventions: every entry point is extern "C", returns int (0 = PRB_OK, < 0 = error) unless
 * noted, takes plain pointers and sizes.  Pointers named *_host / unmarked are caller-owned host
 * buffers (C-contiguous); pointers named *_dev are CUDA device pointers valid on the engine's
 * device.  Host-buffer entry points copy H2D/D2H internally and block until the result is in the
 * caller's buffer.  *_dev entry points only enqueue on the engine's stream (prb_stream) and
 * return; call prb_synchronize (which also reports deferred device-side errors).
 * One engine per process per device; an engine is not re-entrant.  There is NO CPU fallback:
 * prb_create fails when no sm_100-class CUDA device is usable.
 */
#ifndef PYRAD_B200_H
#define PYRAD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PRB_OK               0
#define PRB_ERR_CUDA        -1   /* CUDA runtime error (see prb_last_error) */
#define PRB_ERR_ARG         -2   /* invalid argument */
#define PRB_ERR_STATE       -3   /* call order violated (e.g. line_sum before prepass) */
#define PRB_ERR_RANGE       -4   /* grid segment too large for exact FP32 offsets, or coefficient overflow */
#define PRB_ERR_NODEVICE    -5   /* no usable CUDA device: there is no CPU fallback */
#define PRB_ERR_PEER        -6   /* peer-memory gather: IPC mapping failed or a rank did not arrive */
#define PRB_ERR_PARSE       -7   /* text ingestion: a row or number is not in the expected format */

#define PRB_ABI_VERSION      3

/* prb_line_sum output modes */
#define PRB_OUT_F64          0   /* double per grid point */
#define PRB_OUT_F32          1   /* float per grid point (atmosphere k-matrix rows) */

/* K2 kernel variants (for A/B parity tests and profiling) */
#define PRB_K2_GENERAL       0   /* every staged line through the predicated two-term path */
#define PRB_K2_CLASSED       1   /* per-warp window classes + paired-reciprocal far path (default) */
#define PRB_K2_FARFIELD      2   /* CLASSED, and for windows of >= 256 points the Lorentz wings of lines more than one span length
                                    from a warp's 128/256-point span (and covering it fully) are summed at 16 Chebyshev nodes of
                                    the span and interpolated once per tile; for windows of four tile lengths and more, lines far
                                    from the whole 2048-point tile once per tile.  Interpolation error <= 2e-8 of k (FP64 model of
                                    the algorithm); opt-in -- the default and every headline number are the exact kernel; see
                                    DESIGN.md section 4 */

/* prb_set_option */
#define PRB_OPT_BATCH_LAYERS        1   /* prb_atmosphere: one K1 + one K2 launch per kernel class (default 1) */
#define PRB_OPT_FUSE_SINGLE_LAYER   2   /* single-layer prb_atmosphere: layer physics in K2's epilogue (default 1) */
#define PRB_OPT_RECORD_BUDGET_MB    3   /* device memory for resident per-layer line records; 0 = auto */
#define PRB_OPT_FOLD_TMA            5   /* layer fold: k matrix staged through shared memory by TMA (default 1) or register-held loads (0) */
#define PRB_OPT_SPLIT_TILES         6   /* K2 launches of a few waves: every tile becomes up to 8 work items over parts of its line
                                           range, FP64 partials combined in part order by the CTA that finishes last (default 0).
                                           Removes the idle tail of short launches (strong scaling over small chunks); the
                                           regrouped FP64 sums differ from the unsplit run in the last bits, so the bitwise
                                           shard invariance of the default holds only with the option off */
#define PRB_OPT_POINT_KERNEL        4   /* narrow windows: table-driven k2_point (default 1) or binary-search k2_narrow (0) */

#define PRB_PEER_HANDLE_BYTES      64   /* sizeof(cudaIpcMemHandle_t) */

typedef struct prb_engine prb_engine;

/* ---- lifecycle ------------------------------------------------------------------------- */
int         prb_abi_version(void);
const char *prb_last_error(void);                       /* thread-local, never NULL */
int         prb_create(int device, prb_engine **out);
int         prb_destroy(prb_engine *e);
void       *prb_stream(prb_engine *e);                  /* the engine's cudaStream_t */
int         prb_synchronize(prb_engine *e);             /* stream sync + deferred device status */
/* page-locked host memory (cudaHostAlloc) for line columns / result buffers a caller keeps: copies to and from it run at
 * PCIe speed instead of through the driver's staging buffer; NULL when no CUDA device is usable */
void       *prb_host_alloc(size_t bytes);
int         prb_host_free(void *p);
int         prb_device_info(prb_engine *e, int *sm_count, int *cc_major, int *cc_minor,
                            int *sm_clock_khz, size_t *free_bytes, size_t *total_bytes);
/* Roofline denominators measured on this device (bench.py): FP32 lane-FMAs per second of a packed-FFMA2 and of a scalar
 * FFMA instruction stream, and the float4 copy bandwidth (read + write bytes per second); any pointer may be NULL. */
int         prb_measure_peaks(prb_engine *e, double *ffma2_lane_fma_per_s, double *ffma_lane_fma_per_s,
                              double *copy_bytes_per_s);
int         prb_set_k2_variant(prb_engine *e, int variant, int points_per_thread /* 0 = auto */);
/* windows with W-2 < wm_below use the thread-per-point kernel k2_narrow (0 = never, <0 = default 100) */
int         prb_set_narrow_threshold(prb_engine *e, int64_t wm_below);

/* ---- line list (a1): SoA float64, ascending nu0; group[i] in [0, n_groups) or NULL (all 0) -
 * The list is checked before the call returns (ascending nu0, NaN included; group ids in range -> PRB_ERR_ARG and no
 * list is set) by device kernels over the uploaded columns; the caller's arrays are read once, by the copies. */
int prb_upload_lines(prb_engine *e, int64_t n,
                     const double *nu0, const double *s296,
                     const double *gamma_air, const double *gamma_self,
                     const double *elower, const double *n_air, const double *delta_air,
                     const int32_t *group, int32_t n_groups);

/* Grouped line list (section 8(b): per-group output rows in one pass; pyradClasses.py:350-359, 498-503, 566-576): the
 * host objects hold one line list per isotopologue, each ascending in nu0.  They are uploaded from where they are -- every
 * column argument is a table of n_groups pointers, group g's column has counts[g] entries; no merge sort, no host-side
 * concatenation -- and prb_line_sum_groups returns one
 * cross-section row per group from ONE prepass + ONE line-sum launch (every group walks only its own lines).  Replaces
 * prb_upload_lines; prb_set_grid / prb_layer_prepass / prb_pair_count / prb_line_survey work as before, prb_line_sum and
 * prb_atmosphere need the single ascending list of prb_upload_lines. */
int prb_upload_line_groups(prb_engine *e, int32_t n_groups, const int64_t *counts,
                           const double *const *nu0, const double *const *s296,
                           const double *const *gamma_air, const double *const *gamma_self,
                           const double *const *elower, const double *const *n_air, const double *const *delta_air);

/* Line list straight from HITRAN-online CSV text (section 8(f) row 1; pyradUtilities.py:173-189, 421-448): `text`
 * is the concatenation of the segment files (host memory; rows molec,iso,nu,sw,a,elower,gamma_air,gamma_self,
 * delta_air,n_air; rows starting with '#' are skipped).  Parsed ON THE DEVICE with exact decimal->double
 * conversion (the value float() returns; numbers of more than 19 significant digits included whenever their first 19
 * digits decide the rounding), kept when wave_min < nu < wave_max (strict), duplicate wavenumbers collapse to the
 * last row.  Ascending files (HITRAN's) keep their order; rows in any other order are sorted by wavenumber on the
 * device, the last row of a wavenumber winning wherever it stands (the reference keys a dict by nu).  Replaces
 * prb_upload_lines (single group).  prb_download_lines
 * copies the resulting columns to host buffers (n = prb_line_count entries each; any may be NULL). */
int     prb_ingest_hitran_csv(prb_engine *e, const char *text, int64_t n_bytes, double wave_min, double wave_max,
                              int64_t *n_lines_out);
int     prb_download_lines(prb_engine *e, double *nu0, double *s296, double *einstein_a, double *elower,
                           double *gamma_air, double *gamma_self, double *delta_air, double *n_air);
int64_t prb_line_count(prb_engine *e);                  /* lines on the device; < 0 when none */
/* xsc cross-section table text (two space-separated columns; returnXscFileContents pyradUtilities.py:680-696) parsed
 * on the device: rows that are not exactly two numbers are skipped, as the reference skips them.  capacity = entries
 * the two output arrays can hold (the row count of the text is always enough); n_rows_out = rows kept. */
int     prb_parse_xsc_text(prb_engine *e, const char *text, int64_t n_bytes, int64_t capacity, double *wavenumber,
                           double *cross_section, int64_t *n_rows_out);
int     prb_debug_parse_double(const char *text, int64_t n_bytes, double *value);   /* host-side run of the device parser */

/* ---- grid (a10/a11): point i of the FULL grid sits at range_min + i*res, i in [0, n_total).
 * This engine (rank) owns the contiguous chunk [i_begin, i_end).  Computes every line's
 * arrayIndex = int((nu0 - range_min)/res) (FP64 divide, truncation toward zero) on the device. */
int prb_set_grid(prb_engine *e, double range_min, double res,
                 int64_t n_total, int64_t i_begin, int64_t i_end);

/* ---- K1 (a2-a6, a9 coefficients): per-layer, per-line prepass.
 * Per group g: conc[g] = molecule mole fraction, molmass[g] in g/mol, q_t[g] = Q(T), q_296[g] = Q(296),
 * weight[g] multiplies the group's contribution (1.0 for a cross section; conc*P/1e4/k/T for an
 * absorption coefficient).  window_len = W = len(np.arange(0, cutoff, res)). */
int prb_layer_prepass(prb_engine *e, double T, double P, int32_t n_groups,
                      const double *conc, const double *molmass,
                      const double *q_t, const double *q_296, const double *weight,
                      int64_t window_len);

/* ---- K2 (a7-a10): sum of line shapes into the owned grid chunk; out has i_end-i_begin entries. */
int prb_line_sum(prb_engine *e, double *out_host);
int prb_line_sum_dev(prb_engine *e, void *out_dev, int out_mode);
/* Per-group rows of the last prepass, one K2 launch: out_host [n_groups][i_end-i_begin] row-major, or NULL to leave
 * the rows on the device for prb_layer_spectra_resident. */
int prb_line_sum_groups(prb_engine *e, double *out_host);
/* absCoef / transmittance / Layer.transmission (pyradClasses.py:581-587, 707-716, 784-787) from rows already on the
 * device: k = sum_g sigma_g * group_weight[g] (the rows of the last prb_line_sum_groups) + sum_t xsc_t * xsc_weight[t]
 * (the resident xsc tables; xsc_weight NULL: none).  FP64 host buffers of chunk length; any output may be NULL; the
 * wavenumber axis is linspace(range_min, range_max, n_total) as in prb_atmosphere. */
int prb_layer_spectra_resident(prb_engine *e, const double *group_weight, const double *xsc_weight,
                               double depth_cm, double t_layer, double range_max, const double *radiance_in,
                               double *abs_coef, double *transmittance, double *radiance_out);
int64_t prb_pair_count(prb_engine *e);                  /* accumulations of the last prepass' window on the owned chunk; <0 = error */

/* ---- K1 introspection for parity tests: FP64 per-line values of the last prepass (host buffers,
 * n entries each, any may be NULL): shifted nu, gamma_L, gamma_D, S(T), regime (0 G, 1 L, 2 V), index */
int prb_debug_line_params(prb_engine *e, double *nu_shift, double *gamma_l, double *gamma_d,
                          double *s_t, int32_t *regime, int64_t *index);

/* ---- K3 (a13-a16): fused pointwise layer physics on host buffers, FP64.
 * sigma: n_mol rows of n points (row-major).  weight[m] = conc*P/1e4/k/T.  nu_i = x0 + i*dx for
 * i < n-1 and x_last for i = n-1 (np.linspace semantics; pass the values of Layer.xAxis).
 * Outputs (any may be NULL): abs_coef, transmittance, radiance_out = T*radiance_in + (1-T)*B(nu,t_layer).
 * radiance_in may be NULL when radiance_out is NULL. */
int prb_layer_stream(prb_engine *e, int64_t n, int32_t n_mol, const double *sigma,
                     const double *weight, double depth_cm, double t_layer,
                     double x0, double dx, double x_last,
                     const double *radiance_in,
                     double *abs_coef, double *transmittance, double *radiance_out);

/* planckWavenumber on the same axis convention (pyradPlanck.py:38-44) */
int prb_planck(prb_engine *e, int64_t n, double x0, double dx, double x_last, double temp, double *out);

/* ---- xsc (a17): out[n_out]: zeros, except out[dst0 + j] = src(src0 + j) for j in [0, count), where
 * src(m) = file_y[m] when interp == 0, else np.interp(ax0 + m*adelta, file_x, file_y). */
int prb_xsc_place(prb_engine *e, int64_t n_out, int64_t dst0, int64_t src0, int64_t count,
                  int interp, double ax0, double adelta,
                  int64_t n_file, const double *file_x, const double *file_y, double *out);

/* ---- resident xsc tables (a17 on the device-resident path; pyradClasses.py:466-505, 707-712).  An xsc molecule's cross
 * section is its table, whatever the layer: prb_xsc_resident keeps table `slot` (0 .. 7; an existing slot or the next free
 * one) on the device together with its placement plan -- the arguments of prb_xsc_place, n_out = the grid's n_total --
 * and the engine resamples it onto the owned grid chunk once per grid.  prb_set_xsc_conc gives the tables' mole fractions
 * per layer (L x n_xsc, row-major) for the following prb_atmosphere / prb_gas_cell_host calls with that many layers:
 * every layer's k(nu) then includes  sigma_t(nu) * conc[l][t] * P_l / 1e4 / kB / T_l  (added to the finished line sum
 * inside the line-sum kernel's epilogue).  prb_xsc_clear drops all tables. */
int prb_xsc_resident(prb_engine *e, int32_t slot, int64_t n_out, int64_t dst0, int64_t src0, int64_t count,
                     int interp, double ax0, double adelta,
                     int64_t n_file, const double *file_x, const double *file_y);
int prb_set_xsc_conc(prb_engine *e, int32_t n_layers, int32_t n_xsc, const double *conc);
int prb_xsc_clear(prb_engine *e);
/* A water-vapour continuum in MT_CKD's form for every later prb_atmosphere and prb_gas_cell_host call with n_layers
 * layers, until changed (grid changes keep it).  For layer l (T_l in K, P_l in hPa, x_l = mole_fraction[l] of the
 * continuum's gas) and every point nu of the Planck axis, row l of the k matrix gains, before the fold,
 *   k_c,l(nu) = n_l rho_l R(nu, T_l) [x_l (t_ref/T_l)^n(nu) C_s(nu) + (1 - x_l) C_f(nu)]   in cm^-1,
 *   n_l = x_l P_l / 1e4 / kB / T_l (molecules cm^-3),  rho_l = (P_l / p_ref)(t_ref / T_l),  R(nu, T) = nu tanh(c2 nu / 2T),
 * C_s, C_f = np.interp(nu, table_nu, c_self / c_foreign, left=0, right=0) in cm^2 molecule^-1 (cm^-1)^-1 and
 * n = np.interp(nu, table_nu, t_exp) (clamped at the ends).  Layers with x_l = 0 are left alone.  The table must match
 * the line shape: MT_CKD's coefficients belong to lines cut at 25 cm^-1 with the 25 cm^-1 value subtracted, while this
 * path cuts the lines at 5 P/p0 cm^-1 and adds whatever table it is given.  n_table = 0 clears the continuum (the
 * pointers may then be NULL); otherwise n_table >= 2, table_nu finite and strictly ascending, c_self and c_foreign finite
 * and >= 0, t_exp finite, t_ref and p_ref finite and > 0, n_layers >= 1 and every mole fraction in [0, 1], or PRB_ERR_ARG
 * and the previous setting stays.  A column of another layer count gets PRB_ERR_ARG.  With a continuum, one layer takes
 * the separate fold instead of K2's fused epilogue, and prb_gas_cell_host takes its separate calls; without one, every
 * result is what it was before. */
int prb_set_continuum(prb_engine *e, int64_t n_table, const double *table_nu, const double *c_self,
                      const double *c_foreign, const double *t_exp, double t_ref, double p_ref, int32_t n_layers,
                      const double *mole_fraction);

/* ---- per-layer line ranges.  The reference loads every layer's lines from that layer's own effective range, strictly
 * inside (Isotope.getData -> gatherData(effectiveRangeMin, effectiveRangeMax), pyradClasses.py:350-352,
 * pyradUtilities.py:437-438).  When ONE uploaded list serves a column of layers with different cutoffs, a layer whose
 * cutoff is shorter than a grid step would otherwise pick up a line the reference never loaded for it (a line within one
 * step below rangeMin lands on grid index 0: int() truncates towards zero, pyradClasses.py:390).  With ranges set, layer l
 * of the following prb_atmosphere / prb_gas_cell_host calls (same n_layers) uses only lines with
 * nu_lo[l] < nu0 < nu_hi[l]; n_layers = 0 clears. */
int prb_set_layer_line_range(prb_engine *e, int32_t n_layers, const double *nu_lo, const double *nu_hi);

/* ---- atmosphere (cfg 4): L layers bottom -> top on the owned chunk, everything on the device:
 * per layer K1 + K2 (absorption-coefficient mode, FP32 row of the k matrix), then ONE K3 pass
 * folding I <- T_l*I + (1-T_l)*B(nu, t[l]) with I_0 = B(nu, t_surface).  Per-layer arrays have L
 * entries; per-(layer, group) arrays are L x n_groups row-major.  nu for Planck follows the
 * reference's Layer.xAxis: linspace(range_min, range_max, n_total).
 * Results stay on the device (prb_atmosphere_result_dev) or are copied out (prb_atmosphere_read). */
int prb_atmosphere(prb_engine *e, int32_t n_layers, int32_t n_groups,
                   const double *depth_cm, const double *t_layer, const double *p_layer,
                   const double *conc, const double *molmass, const double *q_t, const double *q_296,
                   const int64_t *window_len, double t_surface, double range_max);
/* One call from HOST line columns to the spectra of one gas cell, with the host->device copies overlapped with the
 * compute: = prb_upload_lines + prb_set_grid + prb_atmosphere(1 layer), bit for bit, but the columns cross PCIe in
 * wavenumber pieces and each piece's prepass and line sum (one wave of K2 tiles) start as soon as it has landed.
 * Combine with prb_set_result_host for results that arrive in host memory the same way (pinned buffers recommended
 * for the inputs too).  Leaves the line list, grid and results on the device like the three separate calls.
 * The line list is validated ON THE DEVICE while it is being used (ascending nu0, group ids in range): on PRB_ERR_ARG
 * from that check the result buffers (device arrays, and the host buffers of prb_set_result_host) hold undefined values.
 * Resident xsc tables (prb_xsc_resident + prb_set_xsc_conc for one layer) are included like in prb_atmosphere. */
int prb_gas_cell_host(prb_engine *e, int64_t n, const double *nu0, const double *s296, const double *gamma_air,
                      const double *gamma_self, const double *elower, const double *n_air, const double *delta_air,
                      const int32_t *group, int32_t n_groups, double range_min, double res, int64_t n_total,
                      int64_t i_begin, int64_t i_end, double depth_cm, double t_layer, double p_layer,
                      const double *conc, const double *molmass, const double *q_t, const double *q_296,
                      int64_t window_len, double t_surface, double range_max);
int prb_atmosphere_result_dev(prb_engine *e, void **radiance_dev, void **transmittance_dev); /* float[chunk] each */
int prb_atmosphere_read(prb_engine *e, double *radiance_host, double *transmittance_host);
int prb_atmosphere_read_f32(prb_engine *e, float *radiance_host, float *transmittance_host);   /* no widening */
/* Zero-copy delivery: register PINNED, 16-byte aligned host buffers (n_points floats each); every following
 * prb_atmosphere also stores its finished spectra there from inside the kernels (tile by tile over PCIe while the
 * line sum is still running), so no read call is needed.  Pass NULL, NULL, 0 to switch it off. */
int prb_set_result_host(prb_engine *e, float *radiance_host, float *transmittance_host, int64_t n_points);
/* stage timing: CUDA events on the engine stream, summed over layers, of the last prb_atmosphere */
int prb_set_timing(prb_engine *e, int enabled);
int prb_atmosphere_timing(prb_engine *e, float *k1_ms, float *k2_ms, float *k3_ms);
int prb_atmosphere_layer_timing(prb_engine *e, int32_t n_layers, float *k1_ms, float *k2_ms);   /* per layer */
int prb_atmosphere_kmatrix_dev(prb_engine *e, void **kmat_dev, int64_t *ld);                 /* float[L][ld] */
int prb_atmosphere_launches(prb_engine *e);              /* kernels launched by the last prb_atmosphere */
/* Hemispheric fluxes and slant radiances of the last column (prb_atmosphere or prb_gas_cell_host), on the owned chunk,
 * from its device-resident k matrix.  For every node i of an angular quadrature (mu[i] in (0, 1], weight[i] > 0,
 * 1 <= n_mu <= 4) the fold I <- T I + (1 - T) B(nu, t[l]), T = exp(-k_l depth_l / mu[i]), runs up from B(nu, t_surface)
 * and down from 0 (a black surface, nothing from above, no solar source; prb_set_flux_boundaries changes the first two,
 * prb_set_solar_source adds the Sun's beam to flux_down, and its reflection to flux_up).
 * Level j is the boundary below layer j: 0 = surface, L = top.
 * flux_up / flux_down: L+1 doubles each, F[j] = 2 pi sum_i weight[i] mu[i] sum_nu I_i(nu, level j) res over this chunk
 * (NaN -- the 0 cm^-1 point -- counts as 0, as in integrateSpectrum, and so does +-inf: next to 0 cm^-1 the reference's
 * negative Doppler widths can make k < 0 and the FP32 transmittance overflow; with wavenumber chunks the ranks' values add up).
 * rad_up_top / rad_down_surface: n_mu x chunk floats each, row-major: the radiance leaving the top along mu[i], and the
 * radiance reaching the surface along mu[i].  Any output may be NULL.  Planck is evaluated as in the column's fold, so
 * mu = 1 reproduces prb_atmosphere's radiance bit for bit.  Under a peer connection the call stays local. */
int prb_atmosphere_fluxes(prb_engine *e, int32_t n_mu, const double *mu, const double *weight,
                          double *flux_up, double *flux_down, float *rad_up_top, float *rad_down_surface);
/* The same fluxes as prb_atmosphere_fluxes (same column, quadrature rules, levels and non-finite rule), split by wavenumber
 * band.  Grid point i belongs to band b when edges[b] <= x_i < edges[b+1], x the column's Planck axis
 * (linspace(range_min, range_max, n_total)); points outside [edges[0], edges[n_bands]) count nowhere, and a band with no
 * points gives zeros.  edges: n_bands + 1 finite values, strictly ascending (n_bands >= 1).  band_up / band_down:
 * [n_bands][L+1] doubles each, this chunk's share, F_b[j] = 2 pi sum_i weight[i] mu[i] sum_{nu in b} I_i(nu, level j) res;
 * either may be NULL.  Only the k-matrix strips that meet a band are read.  The sums are deterministic and independent of
 * the launch grid: repeated calls give the same bits, and so does a band read from a chunk that holds it whole (chunks
 * aligned to 128 points).  Under a peer connection the call stays local. */
int prb_atmosphere_band_fluxes(prb_engine *e, int32_t n_mu, const double *mu, const double *weight,
                               int32_t n_bands, const double *edges, double *band_up, double *band_down);
/* The two boundaries of every later prb_atmosphere_fluxes and prb_atmosphere_band_fluxes call, until changed (independent
 * of the grid; prb_atmosphere keeps them).  Top (level L), every node: I = B(nu, t_top), 0 when t_top = 0.  Surface
 * (level 0), node i: I = eps(nu) B(nu, t_surface) + (1 - eps(nu)) S_i, with eps(x) = np.interp(x, table_nu,
 * table_emissivity) on the Planck axis x (FP64, rounded to FP32; one entry: a constant; n_table = 0: eps = 1 and the
 * pointers may be NULL).  PRB_REFLECT_LAMBERTIAN: S_i = 2 sum_j weight[j] mu[j] I_down_j(nu, 0), the same for every
 * node; PRB_REFLECT_SPECULAR: S_i = I_down_i(nu, 0).  Where eps = 1 the surface value is B(nu, t_surface) bit for bit,
 * and with t_top = 0 the downward results are those without boundaries bit for bit.  (0, NULL, NULL, 0, 0.0) restores
 * a black surface and 0 at the top.  table_nu must be finite and strictly ascending, every emissivity finite and in
 * [0, 1], reflection one of the two constants, t_top finite and >= 0; otherwise PRB_ERR_ARG and the previous setting
 * stays.  prb_atmosphere's own nadir radiance is not affected: its fold always starts from a black surface. */
#define PRB_REFLECT_LAMBERTIAN 0
#define PRB_REFLECT_SPECULAR   1
int prb_set_flux_boundaries(prb_engine *e, int64_t n_table, const double *table_nu, const double *table_emissivity,
                            int32_t reflection, double t_top);
/* The Sun of every later prb_atmosphere_fluxes and prb_atmosphere_band_fluxes call, until changed (independent of the
 * grid; prb_atmosphere keeps it, and its own nadir radiance is not affected).  A collimated beam along mu_sun =
 * cos(solar zenith), absorbed and neither emitted into nor scattered: E(nu, L) = S(nu), E <- E exp(-k_l depth_l / mu_sun)
 * through every layer going down.  S(x) = np.interp(x, table_nu, table_irradiance, left=0, right=0) on the Planck axis x
 * (FP64, rounded to FP32), in W m^-2 (cm^-1)^-1 on a plane normal to the beam.  flux_down[j] and band_down gain
 * mu_sun sum_nu E(nu, j) res at every level.  The surface reflects 1 - eps(nu) of the beam (eps of
 * prb_set_flux_boundaries; none set: eps = 1, nothing reflected): PRB_REFLECT_LAMBERTIAN adds (1 - eps) mu_sun E(nu, 0) / pi
 * to every node's upward start (so rad_up_top includes it); PRB_REFLECT_SPECULAR sends a beam (1 - eps) E(nu, 0) up
 * along mu_sun through the same layer factors, and flux_up and band_up gain mu_sun sum E_up res at every level.  Neither
 * beam is a node: rad_down_surface never changes.  n_table = 0 clears the Sun (the pointers may be NULL, mu_sun is
 * ignored); n_table >= 2 sets it, with table_nu finite and strictly ascending, every irradiance finite and >= 0, and
 * mu_sun in (0, 1]; otherwise PRB_ERR_ARG and the previous setting stays.  An all-zero table gives the results without
 * the Sun bit for bit. */
int prb_set_solar_source(prb_engine *e, int64_t n_table, const double *table_nu, const double *table_irradiance,
                         double mu_sun);
int prb_set_option(prb_engine *e, int option, int64_t value);

/* ---- section 8(f) rows beside the hot path -------------------------------------------------------
 * prb_line_survey: Isotope.createLineSurvey (pyradClasses.py:409-428) for the uploaded lines on the current
 *   grid: out[int((nu0 - rangeMin)/res)] += S296 in line order, bins outside [0, n_out-1] dropped.  Bit-exact.
 * prb_integrate_spectrum: integrateSpectrum (pyradClasses.py:26-29) = sum(nan_to_num(spectrum)) * unitAngle * res
 *   (deterministic pairwise device reduction).
 * prb_atmosphere_integrate: the same integral of the device-resident radiance of the last prb_atmosphere (owned
 *   chunk), plus the plain sum of the total transmittance; either pointer may be NULL.
 * prb_derived_spectra: emissivity 1-T, optical depth -ln T, absorbance log10(1/T) (pyradClasses.py:73-88,
 *   330-340, 596-606) from a transmittance array; any output may be NULL. */
int prb_line_survey(prb_engine *e, int64_t n_out, double *out_host);
int prb_integrate_spectrum(prb_engine *e, int64_t n, const double *spectrum, double unit_angle, double res,
                           double *value);
int prb_atmosphere_integrate(prb_engine *e, double unit_angle, double res, double *radiance_integral,
                             double *transmittance_sum);
int prb_derived_spectra(prb_engine *e, int64_t n, const double *transmittance, double *emissivity,
                        double *optical_depth, double *absorbance);

/* ---- multi-GPU (section 8(e)): wavenumber chunks, one process per GPU on one NVLink/NVSwitch node.
 * The path has no exchange step; the only collective is the all-gather of the finished spectra, and it is
 * fused into the compute step: after prb_peer_connect, prb_atmosphere stores this rank's radiance and
 * transmittance straight into every rank's gather buffer (peer memory, from inside its last kernel) and
 * finishes with a cross-GPU flag barrier.  All ranks must call prb_atmosphere the same number of times.
 *   prb_peer_alloc     allocate this rank's gather buffer (world slots of max_chunk_points floats, two
 *                      fields, double buffered) and export it: handle_out receives PRB_PEER_HANDLE_BYTES
 *   (host side)        exchange the handles between the ranks (any transport; rank order)
 *   prb_peer_connect   handles = world * PRB_PEER_HANDLE_BYTES bytes, rank order
 *   prb_peer_gathered_dev  float[world][ld] radiance / transmittance of the last step, valid on this device
 *                      once the engine's stream has passed the step */
int prb_peer_alloc(prb_engine *e, int rank, int world, int64_t max_chunk_points, void *handle_out);
int prb_peer_connect(prb_engine *e, const void *handles);
int prb_peer_disconnect(prb_engine *e);
int prb_peer_gathered_dev(prb_engine *e, void **radiance_dev, void **transmittance_dev, int64_t *ld);

#ifdef __cplusplus
}
#endif
#endif /* PYRAD_B200_H */
