/*
 * vppstereo_b200.h -- C ABI of the B200-native (sm_100a) VPP + rSGM hot path.
 *
 * This is the drop-in boundary: every entry point replaces one callable of the reference's two native modules
 * (`pyrSGM`, thirdparty/stereo-vision/reconstruction/base/rSGM/pyrSGM.cpp:761-774, and `vpp_core_opt`,
 * vpp_core/vpp_core_opt.pyx) or one Python-level stage of models/rsgm/rsgm.py / vpp_standalone.py.
 * Citations are relative to the reference root; RSGM/ = thirdparty/stereo-vision/reconstruction/base/rSGM/.
 *
 * Conventions
 *   - plain pointers and sizes only; all image / volume pointers are DEVICE pointers unless named *_host;
 *   - every op takes a frame batch: `n` frames stored back to back (frame stride = the natural array size);
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); calls are asynchronous on it;
 *   - no hidden allocation on the data path: ops that need scratch take a caller-provided workspace
 *     (size from the matching *_workspace_bytes query);
 *   - return value: VPPB200_OK or a negative status.  The argument-validation statuses mirror the TypeError
 *     classes of the reference wrapper (RSGM/pyrSGM.cpp:31-35,:206-222,:330-334,:673-677);
 *   - layouts: images row-major [H][W] or [H][W][C] uint8; cost volumes [H][W][D] uint16, d fastest
 *     (RSGM/StereoBMHelper.h:138-141); disparities float32 [H][W].
 * There is no CPU implementation behind this ABI.
 */
#ifndef VPPSTEREO_B200_H
#define VPPSTEREO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VPPB200_OK 0
#define VPPB200_ERR_WIDTH (-1)       /* width % 16 != 0                      (pyrSGM.cpp:31-35)   */
#define VPPB200_ERR_DISP (-2)        /* D % 8 != 0 or D > 256                (pyrSGM.cpp:212-216) */
#define VPPB200_ERR_THREADS (-3)     /* numThreads not in {1,2,4}            (pyrSGM.cpp:218-222) */
#define VPPB200_ERR_UNIQUENESS (-4)  /* uniqueness not in (0,1]              (pyrSGM.cpp:330-334) */
#define VPPB200_ERR_METHOD (-5)      /* sub-pixel method not in {0,1}        (pyrSGM.cpp:673-677) */
#define VPPB200_ERR_WORKSPACE (-6)   /* workspace missing or too small */
#define VPPB200_ERR_ARG (-7)         /* null pointer / non-positive size / unsupported combination */
#define VPPB200_ERR_CUDA (-100)      /* a CUDA runtime call failed; see vppb200_last_cuda_error() */

/* ---- library ------------------------------------------------------------------------------------------ */
const char *vppb200_version(void);
/* name of the last failing CUDA call + cudaGetErrorString, thread-local; "" if none */
const char *vppb200_last_cuda_error(void);
/* Asynchronous failures of earlier launches on the current device that cannot be reported by the launching call: the
 * v-sweep's CTAs hand path state to each other through memory and wait for one another, and so do the rows of the maxDistance
 * wavefront; a wait that times out (a CTA of the cooperative grid not making progress) raises a device flag and lets the grid
 * finish with undefined results instead of trapping the context.  Returns VPPB200_OK, or VPPB200_ERR_CUDA once per incident (flag cleared).  Synchronises the device. */
int vppb200_async_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t vppb200_launch_count(void);
/* 65536-entry table lut[k] = rcp_nz_ss(-2k) (RSGM/StereoBMHelper.cpp:752-756, used by subPixelRefine :1088-1096) as the
 * library currently uses it when a call passes rcp_lut = NULL: by default the FIXED table of Intel's RCPSS approximation
 * (same numbers on every host); with VPPB200_TUNE_RCP_HOST = 1 the table of the HOST CPU's own RCPSS instruction.  Host pointer. */
int vppb200_rcp_lut_host(float *lut_host);

/* Host-side restatement of glibc srand()/rand() (TYPE_3 additive feedback generator, r[i] = r[i-3] + r[i-31]) so that
 * `init_rand(seed)` + scans (vpp_core_opt.pyx:33-35,:93,:102) reproduce the reference's libc pattern stream without
 * touching the process-global libc state.  state: 34 x uint32 owned by the caller.  vppb200_glibc_rand_fill writes
 * n values of rand() % 256 to out_host and advances the state. */
int vppb200_glibc_srand(uint32_t *state34, uint32_t seed);
int vppb200_glibc_rand_fill(uint32_t *state34, uint8_t *out_host, int64_t n);

/* Per-stage device timing of vppb200_compute_rsgm (CUDA events recorded on the call's stream at the stage boundaries).
 * The 8-path aggregation runs as four sweeps (csrc/sgm_sweep.cu): horizontal forward, vertical+diagonal down,
 * vertical+diagonal up, horizontal backward; the last one also produces the WTA / sub-pixel disparities, so the WTA slot
 * only fills on the paths that still materialise the aggregated volume (test tap, shapes the cluster sweep cannot hold,
 * where the whole per-path aggregation is booked on the SGM_H_BWD slot).
 * vppb200_stage_timing(1) enables and resets; vppb200_stage_times synchronises the pending events, writes the
 * accumulated milliseconds per stage to ms_out[VPPB200_N_STAGES] and the number of timed calls to *calls_out. */
#define VPPB200_STAGE_PAD_GRAY 0
#define VPPB200_STAGE_CENSUS 1
#define VPPB200_STAGE_COST 2
#define VPPB200_STAGE_SGM_H_FWD 3
#define VPPB200_STAGE_SGM_V_DOWN 4
#define VPPB200_STAGE_SGM_V_UP 5
#define VPPB200_STAGE_SGM_H_BWD 6
#define VPPB200_STAGE_WTA 7
#define VPPB200_STAGE_MEDIAN_INTERP 8
#define VPPB200_STAGE_TAIL 9
#define VPPB200_N_STAGES 10
int vppb200_stage_timing(int enable);
int vppb200_stage_times(float *ms_out, int *calls_out);

/* Tuning / test hooks (process-wide, not part of the reference's interface).  compute_rsgm aggregates with the
 * four sweeps of csrc/sgm_sweep.cu when a team of resident CTAs can hold the frame's path state in shared memory and
 * with the per-path kernels of csrc/sgm.cu otherwise; results are identical.
 *   VPPB200_TUNE_SGM_MAX_STRIP: upper bound on columns per CTA strip (0 = chosen by the planner); small values force
 *                               many-CTA teams on small frames (parity tests of the halo exchange)
 *   VPPB200_TUNE_SGM_SWEEP:     0 = always use the per-path kernels, 1 = default */
#define VPPB200_TUNE_SGM_MAX_STRIP 0
#define VPPB200_TUNE_SGM_SWEEP 1
#define VPPB200_TUNE_VPP_ROWS 3       /* 0 = VPP rnd by the ordered per-row replay only, 1 = per-pixel replay where possible (default) */
#define VPPB200_TUNE_SGM_CLUSTERS 2   /* upper bound on frames in flight in the v-sweep (0 = all SMs); test hook: forces multi-round teams on small batches */
#define VPPB200_TUNE_VPP_MD_WAVE 5    /* 0 = VPP maxDistance by the serial one-warp-per-(frame, channel) kernel, 1 = row wavefront (default) */
#define VPPB200_TUNE_RCP_HOST 7       /* 0 = sub-pixel reciprocal from the fixed Intel RCPSS table (default), 1 = from the host CPU's RCPSS instruction */
/* Retired keys: accepted, no effect.  Each selected an alternative to the default path that is no longer built. */
#define VPPB200_TUNE_SGM_BYTE_SUMS 4  /* uint8 partial-sum volumes (measured slower) */
#define VPPB200_TUNE_SGM_FUSE_COST 6  /* a forward h-sweep producing the cost volume (measured slower) */
#define VPPB200_TUNE_SGM_V_RED 8      /* 0 = the v-sweeps update S by load + add + store (measured slower than red.global.add) */
#define VPPB200_TUNE_SGM_V_SPLIT 9    /* 0 = one strip width per batch (the planner already keeps one where splitting does not pay) */
#define VPPB200_TUNE_CENSUS_FUSED 10  /* 0 = pad_gray then census (still run wherever the fused kernel does not apply) */
int vppb200_set_tuning(int key, int value);

/* ---- pyrSGM operators ----------------------------------------------------------------------------------- */
/* census5x5_SSE(src u8[H,W], dst u32[H,W], W, H)                       RSGM/pyrSGM.cpp:14, FastFilters.cpp:181-442.
 * Pixels the reference leaves unwritten (rows 0,1,H-2,H-1 and (H-3,{W-16,W-15,W-2,W-1})) are written as 0. */
int vppb200_census5x5(const uint8_t *src, uint32_t *dst, int W, int H, int n, void *stream);

/* costMeasureCensus5x5_xyd_SSE(cl, cr, dsi u16[H,W,D], W, H, D, nthreads) RSGM/pyrSGM.cpp:180, StereoBMHelper.cpp:29-140 */
int vppb200_cost_census5x5_xyd(const uint32_t *cl, const uint32_t *cr, uint16_t *dsi, int W, int H, int D,
                               int num_threads, int n, void *stream);

/* aggregate_SSE(img u8, dsi, dsiAgg, W, H, D, P1, P2min, Alpha, Gamma)     RSGM/pyrSGM.cpp:504, StereoSGM_SSE.hpp:13-515.
 * The reference parses P1..Gamma and then ignores them (pyrSGM.cpp:519 vs :557-560): the effective values are
 * P1=7, P2min=17, Alpha=0.25, Gamma=50.  honor_params=0 reproduces that; honor_params=1 uses the arguments.
 * `img` = the first W*H bytes of the guide image buffer, read as a flat byte stream (pyrSGM.cpp:586-588). */
int vppb200_aggregate(const uint8_t *img, const uint16_t *dsi, uint16_t *dsi_agg, int W, int H, int D,
                      int P1, int P2min, float alpha, int gamma, int honor_params, int n, void *stream);

/* matchWTA_SSE / matchWTARight_SSE(dsiAgg, disp f32[H,W], W, H, D, uniqueness)  RSGM/pyrSGM.cpp:296,:399,
 * StereoBMHelper.cpp:634-750,:893-1015.  First arg-min; uniqueness is validated and otherwise dead, as upstream (the _uniq
 * variants below apply it). */
int vppb200_match_wta(const uint16_t *dsi_agg, float *disp, int W, int H, int D, float uniqueness, int n, void *stream);
int vppb200_match_wta_right(const uint16_t *dsi_agg, float *disp, int W, int H, int D, float uniqueness, int n, void *stream);

/* subPixelRefine(dsi, disp, W, H, D, method)                             RSGM/pyrSGM.cpp:639, StereoBMHelper.cpp:1065-1135.
 * rcp_lut: DEVICE copy of the vppb200_rcp_lut_host table (method 0); NULL = the library's table (see vppb200_rcp_lut_host). */
int vppb200_subpixel_refine(const uint16_t *dsi, float *disp, int W, int H, int D, int method, const float *rcp_lut,
                            int n, void *stream);

/* median3x3_SSE(src f32, dst f32, W, H)                                   RSGM/pyrSGM.cpp:97, FastFilters.cpp:701-757 */
int vppb200_median3x3(const float *src, float *dst, int W, int H, int n, void *stream);

/* ---- compute_rsgm: whole pipeline on device ----------------------------------------------------------------
 * compute_rsgm(left, left_vpp, right_vpp, hints, validhints, dmax, ..., subpixel)   models/rsgm/rsgm.py:250-294.
 * Inputs uint8 [n][H][W][C] (C = 1 or 3; `left` is the adaptive-P2 guide), optional hints/validhints float32
 * [n][H][W] (both NULL = unguided), output float32 [n][H][W].  p1/p2min/alpha/gamma do not exist here because
 * the reference ignores them (vppb200_compute_rsgm_ex honours them on request).  flags: bit0 = subpixel. */
size_t vppb200_rsgm_workspace_bytes(int H, int W, int C, int D, int n);
int vppb200_compute_rsgm(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp,
                         const float *hints, const float *validhints, float *disp_out,
                         int H, int W, int C, int D, int flags, const float *rcp_lut,
                         void *workspace, size_t workspace_bytes, int n, void *stream);

/* The same pipeline in three phases, for callers that overlap neighbouring batches on different streams (the reference
 * has no such interface: it is this library's pipelining of rsgm.py:250-294 across calls).
 *   FRONT: pad + gray + census + Hamming volume (rsgm.py:254-268)   reads the images, writes buffer set `set`
 *   MAIN : 8-path aggregation + WTA left/right (rsgm.py:270-273)    reads / writes buffer set `set`
 *   TAIL : median, interpolation, crop, LR check, speckles, fills (rsgm.py:272-292)  reads set `set`, writes disp_out
 * `phases` = any OR of the three, run in that order on `stream`; the workspace must hold `sets` (1..4) buffer sets
 * (vppb200_rsgm_workspace_bytes_sets).  Ordering between calls on different streams is the caller's job (events);
 * phases == 7 with sets == 1 is vppb200_compute_rsgm.  Image pointers may be NULL when FRONT is not requested, disp_out
 * when TAIL is not; hints/validhints are read by FRONT only. */
#define VPPB200_PHASE_FRONT 1
#define VPPB200_PHASE_MAIN 2
#define VPPB200_PHASE_TAIL 4
size_t vppb200_rsgm_workspace_bytes_sets(int H, int W, int C, int D, int n, int sets);
int vppb200_compute_rsgm_phases(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp,
                                const float *hints, const float *validhints, float *disp_out,
                                int H, int W, int C, int D, int flags, const float *rcp_lut,
                                void *workspace, size_t workspace_bytes, int n, void *stream,
                                int phases, int sets, int set);

/* Stage taps of the same pipeline for tests (any pointer may be NULL): padded census L/R u32 [n][Hp][Wp], aggregated
 * volume u16 [n][Hp][Wp][D], left/right disparities after median+interpolation+clip f32 [n][Hp][Wp].  Set before the
 * call, valid after the stream is synchronised. */
typedef struct {
    uint32_t *census_l, *census_r;
    uint16_t *dsi_agg;
    float *disp_l, *disp_r;
} vppb200_rsgm_taps;
int vppb200_compute_rsgm_tapped(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp,
                                const float *hints, const float *validhints, float *disp_out,
                                int H, int W, int C, int D, int flags, const float *rcp_lut,
                                void *workspace, size_t workspace_bytes, int n, void *stream,
                                const vppb200_rsgm_taps *taps);

/* ---- honoured SGM parameters (an opt-in the reference does not have: it parses P1..Gamma and overwrites them with 7, 17,
 * 0.25, 50, RSGM/pyrSGM.cpp:519 vs :557-560).  Semantics: the reference's StereoSGM recursion with the parameters as arguments
 * (RSGM/StereoSGM_SSE.hpp:13-515), P2 = max(p2min, (int32)(-alpha * |I_p - I_pr| + gamma)) in float32 with the two operations
 * rounded separately (RSGM/StereoSGM.hpp:92-99).
 *   vppb200_compute_rsgm_ex: vppb200_compute_rsgm_phases + taps (phases == 7 only, as vppb200_compute_rsgm_tapped) + params.
 *       params == NULL: the reference's effective values (7, 17, 0.25, 50) -- exactly what the other entry points do.  Every
 *       phase of one batch must be called with the same params and hints (they select the layout of the cost volume).
 *   vppb200_sgm_band_ex: vppb200_sgm_band + params; refuses parameters outside the sweep domain (there is no per-path band path).
 *   vppb200_sgm_params_fast: 1 = the four sweeps compute these parameters, 0 = compute_rsgm falls back to the per-path kernels,
 *       VPPB200_ERR_ARG = invalid.  guided: costs modulated by hints (up to 240) instead of plain Hamming costs (up to 24).
 * Validation (before any CUDA call, VPPB200_ERR_ARG otherwise): 0 <= p1, p2min, gamma <= 65535; alpha finite and >= 0, so that
 * P2 lies in [p2min, P2max], P2max = max(p2min, gamma).
 * Sweep domain, Cmax = 24 (Hamming) or 240 (guided): p1 <= p2min, P2max - p1 <= 255 and Cmax + P2max <= 4095.  Inside it the four
 * sweeps run as for the default parameters (same speed, no saturation reachable).  Outside it the aggregation runs on the
 * saturating per-path kernels (8 launches, each a read-modify-write of the whole aggregated volume: several times slower),
 * bit-exact with the recursion including its uint16 saturation.  Parameters are kernel arguments: calls with different
 * parameters may run concurrently on different streams. */
typedef struct {
    int p1;
    int p2min;
    float alpha;
    int gamma;
} vppb200_sgm_params;
int vppb200_compute_rsgm_ex(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp,
                            const float *hints, const float *validhints, float *disp_out,
                            int H, int W, int C, int D, int flags, const float *rcp_lut,
                            void *workspace, size_t workspace_bytes, int n, void *stream,
                            int phases, int sets, int set, const vppb200_rsgm_taps *taps,
                            const vppb200_sgm_params *params);
int vppb200_sgm_params_fast(const vppb200_sgm_params *params, int guided);

/* ---- uniqueness ratio of the winner-takes-all (an opt-in: the reference computes its uniqueness test and then overwrites the
 * result, RSGM/StereoBMHelper.cpp:717,:745,:981,:1009, so every other entry point keeps the plain first arg-min).
 * Candidates of a pixel, from the final aggregated volume S: left view c[d] = S[y][x][d], end = min(D-1, x); right view
 * c[k] = S[y][x+k][k], end = min(D-1, W-1-x).  b = the first arg-min (as without the test); c2 = min{c[d] : 0 <= d <= end,
 * |d - b| >= 2} (the neighbours b +- 1 are part of the same minimum); f = (uint32)(1024.0f * uniqueness).  The pixel is accepted
 * when no such d exists (end <= 1, or end == 2 with b == 1) or when 1024 * c[b] <= f * c2 (exact 32-bit arithmetic).  Accepted
 * pixels are exactly what the plain WTA gives (left: including the sub-pixel step); a rejected pixel's raw disparity is -10.0f in
 * both views at every column, which the rest of compute_rsgm treats as any other invalid pixel.
 * uniqueness must be finite with 0 < uniqueness <= 1, otherwise VPPB200_ERR_UNIQUENESS before any CUDA call.  uniqueness == 1
 * (f = 1024) accepts every pixel and runs exactly the kernels of the plain entry point.
 *   vppb200_match_wta_uniq / vppb200_match_wta_right_uniq: vppb200_match_wta / _right with the test.
 *   vppb200_compute_rsgm_uniq: vppb200_compute_rsgm_ex + uniqueness, read by MAIN (every phase of one batch must pass the same
 *       value; it is validated on every call).  The work is booked on the SGM_H_BWD stage (WTA where the volume is materialised).
 *   vppb200_sgm_band_uniq: vppb200_sgm_band_guided + uniqueness, read by phase 16. */
int vppb200_match_wta_uniq(const uint16_t *dsi_agg, float *disp, int W, int H, int D, float uniqueness, int n, void *stream);
int vppb200_match_wta_right_uniq(const uint16_t *dsi_agg, float *disp, int W, int H, int D, float uniqueness, int n, void *stream);
int vppb200_compute_rsgm_uniq(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp,
                              const float *hints, const float *validhints, float *disp_out,
                              int H, int W, int C, int D, int flags, const float *rcp_lut,
                              void *workspace, size_t workspace_bytes, int n, void *stream,
                              int phases, int sets, int set, const vppb200_rsgm_taps *taps,
                              const vppb200_sgm_params *params, float uniqueness);

/* ---- per-pixel match info of the left view (an opt-in the reference does not have: its compute_rsgm returns a dense map in which
 * a measured disparity and a hole filled by _interpolate_background, models/rsgm/rsgm.py:184-227, look the same).  Maps are cropped
 * [n][H][W] like disp_out.  With the stages of compute_rsgm (rsgm.py:250-294) named
 *   m    = the left map after WTA (with the uniqueness test where it is honoured), sub-pixel step and median3x3, padded frame;
 *   c    = max(_linear_interpolate(m), 0), cropped;  mask = _left_right_check(c, c_right);  u = uint8(c with mask == 128 set to 0);
 *   s    = filterSpeckles(u),
 * state uint8 is the code of the first rule that applies, in this order:
 *   VPPB200_STATE_NO_MATCH     c == 0 (no positive WTA winner, uniqueness-rejected, or not positive after the median, and not filled
 *                              by the gap interpolation)
 *   VPPB200_STATE_LR_REJECTED  mask == 128 (includes a match that points outside the right image)
 *   VPPB200_STATE_BELOW_ONE    u == 0 (0 < c < 1, truncated by astype(uint8))
 *   VPPB200_STATE_SPECKLE      s == 0
 *   VPPB200_STATE_INTERPOLATED m <= 0 (the value came from _linear_interpolate)
 *   VPPB200_STATE_MATCHED      otherwise (s > 0 and m > 0).
 * Codes 2..5 are exactly the pixels whose disparity comes from the background fill (or stays 0 where the fill finds nothing).
 * cost, rival uint16, from the final aggregated volume S at the padded pixel (y + pad_top, x + pad_left): with end = min(D-1, x +
 * pad_left) and b = the first arg-min over 0..end, cost = S[b] and rival = min{S[d] : 0 <= d <= end, |d - b| >= 2}, 65535 when no
 * such d exists -- the c[b] and c2 of the uniqueness block above, reported whether or not the test is honoured (and equal either
 * way).  Turning the info on changes no disparity.
 *   vppb200_rsgm_info_workspace_bytes: vppb200_rsgm_workspace_bytes_sets + per-set padded cost / rival maps (they cross the
 *       MAIN -> TAIL boundary like the raw disparities).
 *   vppb200_compute_rsgm_info: vppb200_compute_rsgm_uniq (same arguments, taps included) + the three outputs, all required
 *       (VPPB200_ERR_ARG otherwise); every phase of one batch must pass the same pointers.  MAIN fills the set's cost / rival
 *       maps, TAIL writes state_out, cost_out and rival_out (ordered like disp_out).  A workspace smaller than the info layout:
 *       VPPB200_ERR_WORKSPACE. */
#define VPPB200_STATE_MATCHED 0
#define VPPB200_STATE_INTERPOLATED 1
#define VPPB200_STATE_NO_MATCH 2
#define VPPB200_STATE_LR_REJECTED 3
#define VPPB200_STATE_BELOW_ONE 4
#define VPPB200_STATE_SPECKLE 5
size_t vppb200_rsgm_info_workspace_bytes(int H, int W, int C, int D, int n, int sets);
int vppb200_compute_rsgm_info(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp,
                              const float *hints, const float *validhints, float *disp_out,
                              int H, int W, int C, int D, int flags, const float *rcp_lut,
                              void *workspace, size_t workspace_bytes, int n, void *stream,
                              int phases, int sets, int set, const vppb200_rsgm_taps *taps,
                              const vppb200_sgm_params *params, float uniqueness,
                              uint8_t *state_out, uint16_t *cost_out, uint16_t *rival_out);

/* ---- one frame split into row bands over several GPUs (SURVEY.md 8e: an oversized frame) -------------------------------
 * compute_rsgm (models/rsgm/rsgm.py:250-294) as three calls so that the aggregation -- the 2.2 GB of volumes of a Middlebury
 * frame -- runs band by band on different GPUs, EXACTLY (unlike the reference's approximate StripedStereoSGM,
 * RSGM/StereoSGM.h:116-133): the vertical / diagonal sweeps of a band continue from the row state the neighbouring band exported.
 *   vppb200_rsgm_front_census: pad + RGB2GRAY + census 5x5 of the WHOLE frame (rsgm.py:254-262,:8-28) ->
 *       guide uint8 [Hp*Wp] (the first Hp*Wp bytes of the padded `left`), census_l / census_r uint32 [Hp][Wp]
 *   vppb200_sgm_band: rows [row0, row0 + rows) of the padded frame.  phases (bit mask, queued in this order):
 *       1 Hamming volume of the band, 2 h-sweep forward, 4 v-sweep down, 8 v-sweep up, 16 h-sweep backward + WTA / sub-pixel.
 *       cost_band: uint8 layout-T volume of the band (vppb200_banded_dims: volume_bytes_per_row * rows bytes), S_band twice that.
 *       state_in / state_out: the row state of the three vertical / diagonal paths (state_words uint32 each): phase 4 of a band
 *       with row0 > 0 reads state_in = what phase 4 of the band above wrote to its state_out; phase 8 of a band that does not end
 *       at Hp reads state_in = state_out of phase 8 of the band below.  dl_band / dr_band: float32 [rows][Wp] raw disparities.
 *   vppb200_rsgm_tail: median .. background fill (rsgm.py:273-292) on the gathered raw maps dl, dr float32 [Hp][Wp] -> disp_out
 *       float32 [H][W] (flags bit 0: sub-pixel).  dl / dr are read only.
 * workspace: vppb200_banded_workspace_bytes, private to one call at a time. */
size_t vppb200_banded_workspace_bytes(int H, int W, int C, int D);
int vppb200_banded_dims(int H, int W, int C, int D, int *Hp, int *Wp, int64_t *state_words, int64_t *volume_bytes_per_row);
int vppb200_rsgm_front_census(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp, uint8_t *guide,
                              uint32_t *census_l, uint32_t *census_r, int H, int W, int C, int D, void *workspace,
                              size_t workspace_bytes, void *stream);
int vppb200_sgm_band(const uint8_t *guide, const uint32_t *census_l, const uint32_t *census_r, uint8_t *cost_band,
                     uint16_t *S_band, int H, int W, int C, int D, int row0, int rows, int phases, const uint32_t *state_in,
                     uint32_t *state_out, float *dl_band, float *dr_band, const float *rcp_lut, void *workspace,
                     size_t workspace_bytes, void *stream);
int vppb200_sgm_band_ex(const uint8_t *guide, const uint32_t *census_l, const uint32_t *census_r, uint8_t *cost_band,
                        uint16_t *S_band, int H, int W, int C, int D, int row0, int rows, int phases, const uint32_t *state_in,
                        uint32_t *state_out, float *dl_band, float *dr_band, const float *rcp_lut, void *workspace,
                        size_t workspace_bytes, void *stream, const vppb200_sgm_params *params);
/*   vppb200_sgm_band_guided: vppb200_sgm_band_ex + guided matching (rsgm.py:115-127, the hints / validhints of
 *       vppb200_compute_rsgm): hints, validhints float32 [H][W], the WHOLE unpadded frame.  Both NULL: exactly vppb200_sgm_band_ex;
 *       exactly one NULL: VPPB200_ERR_ARG.  With hints, phase 1 modulates the band's volume (rows of the padded frame map to hint
 *       rows row0 + r - pad_top) and params must lie in the guided sweep domain (Cmax = 240, see vppb200_sgm_params_fast).  Every
 *       phase of every band of one frame must be called with the same params and hint nullness (they select the sweeps' state
 *       representation); hints are only read by phase 1.  Arguments are validated before any CUDA call. */
int vppb200_sgm_band_guided(const uint8_t *guide, const uint32_t *census_l, const uint32_t *census_r, uint8_t *cost_band,
                            uint16_t *S_band, int H, int W, int C, int D, int row0, int rows, int phases, const uint32_t *state_in,
                            uint32_t *state_out, float *dl_band, float *dr_band, const float *rcp_lut, void *workspace,
                            size_t workspace_bytes, void *stream, const vppb200_sgm_params *params, const float *hints,
                            const float *validhints);
/*   vppb200_sgm_band_uniq: see the uniqueness block above. */
int vppb200_sgm_band_uniq(const uint8_t *guide, const uint32_t *census_l, const uint32_t *census_r, uint8_t *cost_band,
                          uint16_t *S_band, int H, int W, int C, int D, int row0, int rows, int phases, const uint32_t *state_in,
                          uint32_t *state_out, float *dl_band, float *dr_band, const float *rcp_lut, void *workspace,
                          size_t workspace_bytes, void *stream, const vppb200_sgm_params *params, const float *hints,
                          const float *validhints, float uniqueness);
int vppb200_rsgm_tail(float *dl, float *dr, float *disp_out, int H, int W, int C, int D, int flags, void *workspace,
                      size_t workspace_bytes, void *stream);

/* ---- vpp_core_opt operators ---------------------------------------------------------------------------------
 * virtual_projection_scan_rnd(l, r, g, width, height, channels, uniform_color, wsize, direction, c, c_occ, g_occ,
 *                             discard_occluded, interpolate) -> #hints                vpp_core_opt.pyx:53-131
 * l, r uint8 [n][H][W][C] are modified in place; g float32 [n][H][W] (0 = no hint); g_occ uint8 [n][H][W].
 * arith: 0 = Cython arithmetic (c as float32, vpp_core_opt.pyx), 1 = numba arithmetic (all float64,
 *        vpp_standalone.py:243-369; round half to even).
 * The reference draws the pattern from libc rand() / numba's generator while scanning; here the caller passes the
 * pre-drawn values: pattern[] (uint8) holds all frames' streams, frame f starts at pattern_offsets[f] (int64, n+1
 * entries) and is consumed in the reference's call order (pyx:92-93,:101-102).
 * pattern == NULL selects on-device pattern generation instead: value = hash(rng_seed, frame, stream position) & 255
 * (counter based, no pattern memory; pattern_offsets may then be NULL too).
 * n_hints_out: int32 [n] device, may be NULL. */
size_t vppb200_vpp_workspace_bytes(int H, int W, int C, int n);
int vppb200_vpp_scan_rnd(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color, int wsize,
                         int direction, double c, double c_occ, const uint8_t *g_occ, int discard_occluded,
                         int interpolate, int arith, const uint8_t *pattern, const int64_t *pattern_offsets,
                         uint64_t rng_seed, int32_t *n_hints_out, void *workspace, size_t workspace_bytes, int n, void *stream);

/* Row-band form of the rnd scan (SURVEY.md 8e: an oversized frame split across GPUs): only the image rows
 * [row_begin, row_end) of l and r are produced, every other row is left untouched.  Exact: a blend that writes image row yy
 * only reads row yy of the same channel, and the stream position of every draw is a closed form of the full hint map g (which
 * every band reads whole), so the union of disjoint bands equals the full scan bit for bit. */
int vppb200_vpp_scan_rnd_rows(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color, int wsize,
                              int direction, double c, double c_occ, const uint8_t *g_occ, int discard_occluded,
                              int interpolate, int arith, const uint8_t *pattern, const int64_t *pattern_offsets,
                              uint64_t rng_seed, int row_begin, int row_end, int32_t *n_hints_out, void *workspace,
                              size_t workspace_bytes, int n, void *stream);

/* virtual_projection_scan_max_dist(l, r, g, width, height, channels, uniform_color, wsize, wsize_agg_x, wsize_agg_y,
 *                                  direction, c, c_occ, g_occ, discard_occluded, interpolate) -> #hints  pyx:133-341
 * Workspace: vppb200_vpp_max_dist_workspace_bytes (adds the per-hint dependency table of the row-wavefront kernel);
 * with only vppb200_vpp_workspace_bytes the call still works but runs the hints of a (frame, channel) one after another. */
size_t vppb200_vpp_max_dist_workspace_bytes(int H, int W, int C, int wsize, int wsize_agg_y, int n);
int vppb200_vpp_scan_max_dist(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color, int wsize,
                              int wsize_agg_x, int wsize_agg_y, int direction, double c, double c_occ,
                              const uint8_t *g_occ, int discard_occluded, int interpolate, int arith,
                              int32_t *n_hints_out, void *workspace, size_t workspace_bytes, int n, void *stream);

/* The adaptive patches of vpp() (TPAMI extension, numba twin only: vpp_standalone.py:6-11 distance-based patch size,
 * :371-394 _bilateral_filling, guards :153-154 / :334-335).  The scans take two optional device operands:
 *   filled_g          float32 [n][H][W], the output of vppb200_bilateral_filling: a patch pixel is projected (and, in rnd mode,
 *                     its pattern value drawn) only where |g[y,x] - filled_g[yy,xx]| < 0.1 (float64); NULL = always
 *   patch_thresholds  float32 [n][wsize-1], ascending: patch size of a hint = 1 + #{k : g >= thr[k]} (the caller tabulates the
 *                     reference's float32-ratio / libm-pow / round-half-even size function into these steps, so the device
 *                     evaluates no pow()); NULL = wsize for every hint
 * vppb200_bilateral_filling: gray = uint8 context image [n][H][W]; weights = DEVICE float64 [(2p+1)^2][256] table of
 * exp(-((yw^2+xw^2)/(2 o_xy^2) + di^2/(2 o_i^2))) indexed by (patch offset, |intensity difference|), tabulated by the caller
 * with the host libm (numba calls the same function); th = bilateral_th. */
int vppb200_bilateral_filling(const float *dmap, const uint8_t *gray, float *out, int W, int H, int n_patch,
                              const double *weights, double th, int n, void *stream);
int vppb200_vpp_scan_rnd_adaptive(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color, int wsize,
                                  int direction, double c, double c_occ, const uint8_t *g_occ, int discard_occluded,
                                  int interpolate, int arith, const uint8_t *pattern, const int64_t *pattern_offsets,
                                  uint64_t rng_seed, const float *filled_g, const float *patch_thresholds, int n_thresholds,
                                  int32_t *n_hints_out, void *workspace, size_t workspace_bytes, int n, void *stream);
int vppb200_vpp_scan_max_dist_adaptive(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color,
                                       int wsize, int wsize_agg_x, int wsize_agg_y, int direction, double c, double c_occ,
                                       const uint8_t *g_occ, int discard_occluded, int interpolate, int arith,
                                       const float *filled_g, const float *patch_thresholds, int n_thresholds,
                                       int32_t *n_hints_out, void *workspace, size_t workspace_bytes, int n, void *stream);

/* The gray context image of vppb200_bilateral_filling from the un-projected left image (vpp_standalone.py:414-417):
 * src uint8 [n][H][W][C] -> gray uint8 [n][H][W]; C = 3: cv2.cvtColor(BGR2GRAY) in OpenCV's 15-bit fixed point
 * (B*3735 + G*19235 + R*9798 + 16384) >> 15; any other C: the first channel. */
int vppb200_bgr2gray(const uint8_t *src, uint8_t *gray, int W, int H, int C, int n, void *stream);

/* The patch_thresholds operand of the adaptive scans, computed on the device (no host round trip).  The reference's size is
 *   size(d) = round(float64(ratio) ** (1/gamma) * (wsize-1) + 1)  (round half to even),
 *   ratio   = float32(float32(d) - dmin) / float32(dmax - dmin),  dmin / dmax = min / max of the frame's hints (g > 0).
 * It splits exactly in two:
 *   host   -- size is a non-decreasing function of the float32 ratio alone, so for k = 2..wsize there is a smallest float32
 *             ratio R_k in [0, 1] with size >= k; the caller tabulates ratio_steps = {R_2 .. R_wsize} (float32 [wsize-1], DEVICE)
 *             once per (wsize, gamma) with the host's libm -- the only evaluation of pow();
 *   device -- per frame (one CTA), dmin / dmax over g > 0, then thr[k-2] = the smallest float32 d in [dmin, dmax] with
 *             ratio(d) >= R_k (ratio with float32 round-to-nearest subtraction and division), by bisection on the bit patterns.
 * patch_thresholds float32 [n][wsize-1]: +inf for a frame without hints (never read) and for a frame whose hints all have one
 * value (dmin == dmax, where the reference raises ZeroDivisionError: patch size 1, a defined result); the latter also sets
 * status[f] = 1 (int32 [n] device, entries of other frames untouched: the caller clears it; may be NULL).  wsize == 1: no
 * thresholds (ratio_steps / patch_thresholds may be NULL), only the status. */
int vppb200_distance_patch_thresholds(const float *g, int W, int H, const float *ratio_steps, int wsize, float *patch_thresholds,
                                      int32_t *status, int n, void *stream);

/* gt_reshape(gt f32[H,W]) -> f32[N,4] = (x, y, d, 1) in raster order           vpp_core_opt.pyx:352-371.
 * out must hold W*H rows; count_out int32 [1] device. */
int vppb200_gt_reshape(const float *gt, int W, int H, float *out, int32_t *count_out, void *workspace,
                       size_t workspace_bytes, void *stream);

/* ---- occlusion mask for VPP: occlusion_heuristic(dmap, rx=9, ry=7, l=2, g=0.4375, th_conf=1, th_filter=0.1)
 * -> (dmap, conf_map)                                                                        filter.py:246-292
 * (left_warp :7-48, weighted_conf :113-164, filter :167-194, left_unwarp :50-79, conf_unwarp :81-111,
 * interpolate_disparity(dmap, 3) :196-243).  test.py:154 passes the sparse hints and uses [1] as g_occ.
 * dmap float32 [n][H][W] (0 = no hint); dmap_out float32 / conf_out uint8 (0 = visible hint, 1 elsewhere), either may
 * be NULL.  rx, ry are the un-halved radii as in the reference signature. */
size_t vppb200_occlusion_workspace_bytes(int H, int W, int n);
int vppb200_occlusion_heuristic(const float *dmap, float *dmap_out, uint8_t *conf_out, int W, int H, int rx, int ry,
                                double l, double g, double th_conf, double th_filter, void *workspace,
                                size_t workspace_bytes, int n, void *stream);

/* ---- hand-off to the networks (test.py:179-200): uint8 [n][H][W][C] -> float32 [n][C][H+pt+pb][W+pl+pr],
 * value = float32(u8 / 255.0) (test.py:179-180), replicate padding as F.pad(..., mode='replicate') (test.py:192-197). */
int vppb200_u8hwc_to_f32chw(const uint8_t *src, float *dst, int H, int W, int C, int pad_top, int pad_bottom,
                            int pad_left, int pad_right, int n, void *stream);

/* The other direction, test.py:158-159 and :210-212: float32 [n][C][H][W] in [0,1] -> uint8 [n][H][W][C] = (uint8)(255.0f * v)
 * (float32 product, truncation), so the loader's normalised tensors reach vpp() / compute_rsgm() without a host hop. */
int vppb200_f32chw_to_u8hwc(const float *src, uint8_t *dst, int H, int W, int C, int n, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* VPPSTEREO_B200_H */
