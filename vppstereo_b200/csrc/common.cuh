// common.cuh -- shared helpers for the sm_100a kernels behind include/vppstereo_b200.h
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/vppstereo_b200.h"

namespace vppb200 {

// kernel-launch accounting (vppb200_launch_count) and CUDA error capture (vppb200_last_cuda_error)
void note_launch(int k = 1);
int cuda_fail(const char *what, cudaError_t e);

#define VPP_CUDA_TRY(expr)                                              \
    do {                                                                \
        cudaError_t _e = (expr);                                        \
        if (_e != cudaSuccess) return ::vppb200::cuda_fail(#expr, _e);  \
    } while (0)

// check the launch that was just issued
#define VPP_LAUNCH_CHECK(name)                                          \
    do {                                                                \
        ::vppb200::note_launch();                                       \
        cudaError_t _e = cudaGetLastError();                            \
        if (_e != cudaSuccess) return ::vppb200::cuda_fail(name, _e);   \
    } while (0)

static inline int cdiv(long a, long b) { return (int)((a + b - 1) / b); }

struct RsgmDims {
    int H, W, C, D;        // user frame
    int pl, pr, pt, pb;    // BORDER_REFLECT padding to multiples of 16 (models/rsgm/rsgm.py:254-256)
    int Hp, Wp;
};

static inline RsgmDims make_dims(int H, int W, int C, int D)
{
    RsgmDims d;
    d.H = H; d.W = W; d.C = C; d.D = D;
    int pad_h = (((H / 16) + 1) * 16 - H) % 16, pad_w = (((W / 16) + 1) * 16 - W) % 16;
    d.pl = pad_w / 2; d.pr = pad_w - d.pl; d.pt = pad_h / 2; d.pb = pad_h - d.pt;
    d.Hp = H + pad_h; d.Wp = W + pad_w;
    return d;
}

// The four SGM penalties (RSGM/StereoSGM.h:33-47).  The reference's effective values are P1 = 7, P2min = 17, alpha = 0.25,
// gamma = 50 (RSGM/pyrSGM.cpp:557-560); callers that honour their own parameters pass them through vppb200_sgm_params.
struct SgmParams {
    int P1, P2min, gamma;
    float alpha;
};
static inline SgmParams default_sgm_params() { return SgmParams{7, 17, 50, 0.25f}; }

// adaptP2 (RSGM/StereoSGM.hpp:92-99): (sint32)(-alpha * |I_p - I_pr| + gamma), clamped below by P2min.  Two separately rounded
// float operations, as the reference's expression compiles without contraction; the only evaluation of P2 in the library.
__device__ __forceinline__ int adapt_p2(const SgmParams &p, int ip, int ipr)
{
    const int r = (int)__fadd_rn(__fmul_rn(-p.alpha, (float)abs(ip - ipr)), (float)p.gamma);
    return r < p.P2min ? p.P2min : r;
}

// ---- uniqueness ratio of the winner-takes-all (opt-in; semantics in include/vppstereo_b200.h) ----------------------------
// uf = (uint32)(1024.0f * u).  UNIQ_OFF (u = 1) accepts every pixel: the launchers then run the plain WTA instantiations.
static constexpr uint32_t UNIQ_OFF = 1024u;

// Accept the pixel whose first arg-min is key = (cost << 16 | b) over the candidates [0, end], c2 = the least cost of a rival
// (|d - b| >= 2)?  Whether a rival exists at all is decided by b and end alone, so c2 may hold a genuine 65535 cost: 0xFFFF in
// the callers' running minima is only the identity of min, never read as "no rival".
__device__ __forceinline__ bool uniq_accept(uint32_t key, uint32_t c2, int end, uint32_t uf)
{
    const int b = (int)(key & 0xFFFFu);
    const bool rival = end >= 3 || (end == 2 && b != 1);
    return !rival || 1024u * (key >> 16) <= uf * c2;
}

// is candidate d a rival of the first arg-min b inside [0, end]?
__device__ __forceinline__ bool uniq_rival(int d, int b, int end) { return d <= end && (unsigned)(d - b + 1) > 2u; }

// One right-view target absorbs its candidate key = (c << 16 | k).  A target sees its candidates in descending k (it takes slot k
// at column t + k of a sweep x = W-1 .. 0), so the least rival cost is kept online: best = the first arg-min so far (as the plain
// WTA), fr = far | rest << 16 with far = min over absorbed k' with |k' - b| >= 2 and rest = min over the absorbed candidates but
// the most recent, last = the most recent cost.  A new best k has only k + 1 (the most recent) as a neighbour among the absorbed
// ones, so its far is the old rest.  Empty state: best = 0xFFFFFFFF, fr = 0xFFFFFFFF, last = 0xFFFF (absorbing the invalid key
// 0xFFFFFFFF keeps it empty).
__device__ __forceinline__ void uniq_absorb(uint32_t &best, uint32_t &fr, uint32_t &last, uint32_t key)
{
    const uint32_t c = key >> 16;
    const bool better = key < best;
    const bool rival = (best & 0xFFFFu) >= (key & 0xFFFFu) + 2u;
    const uint32_t v = __vminu2(fr, (last << 16) | (rival ? c : 0xFFFFu));
    fr = better ? ((v & 0xFFFF0000u) | (fr >> 16)) : v;
    best = better ? key : best;
    last = c;
}

// ---- stage launchers (defined in the .cu files, all asynchronous on `st`) -------------------------------
int launch_pad_gray(const uint8_t *src, uint8_t *gray, const RsgmDims &d, int n, cudaStream_t st);
int launch_pad_flatbytes(const uint8_t *src, uint8_t *guide, const RsgmDims &d, int n, cudaStream_t st);
int launch_census(const uint8_t *src, uint32_t *dst, int W, int H, int n, cudaStream_t st);
int launch_census_fused(const uint8_t *src, uint32_t *dst, const RsgmDims &d, int n, cudaStream_t st);   // pad + gray + census, 1 = n/a
int launch_cost_u16(const uint32_t *cl, const uint32_t *cr, uint16_t *dsi, int W, int H, int D, int n, cudaStream_t st);
int launch_cost_u8(const uint32_t *cl, const uint32_t *cr, uint8_t *dsi, int W, int H, int D, int n, cudaStream_t st);
int launch_guided_u8(uint8_t *dsi, const float *hints, const float *valid, const RsgmDims &d, int n, cudaStream_t st);
// saturating 8-path aggregation, any parameters: CT = uint16_t (aggregate_SSE) or uint8_t (compute_rsgm without the sweeps)
template <typename CT>
int launch_aggregate_generic(const uint8_t *img, const CT *dsi, uint16_t *S, int W, int H, int D, const SgmParams &p, int n,
                             cudaStream_t st);
// sgm_sweep.cu: layout-T cost volume + 4-sweep aggregation with on-chip path state (cluster per frame)
bool aggregate_tile_supported(int W, int H, int D, int n);
// do the sweeps compute these parameters exactly?  plain_costs: Hamming costs (<= 24), otherwise guided costs (<= 240)
bool sweep_params_supported(const SgmParams &p, bool plain_costs);
size_t tile_volume_elems(int W, int H, int D, int n);
// guided modulation of the tiled cost volume (models/rsgm/rsgm.py:115-127), fused into the cost kernel: hints / valid float32
// [n][H][W] of the user frame (hints == NULL: plain Hamming costs); pl / pt / W / H place the user frame inside the padded one
struct GuideOps {
    const float *hints, *valid;
    int pl, pt, W, H;
};
static inline GuideOps guide_ops(const float *hints, const float *valid, const RsgmDims &d)
{
    return GuideOps{hints, valid, d.pl, d.pt, d.W, d.H};
}
int launch_cost_tile(const uint32_t *cl, const uint32_t *cr, uint8_t *cost, int W, int H, int D, int n, const GuideOps &gd,
                     cudaStream_t st);
int launch_cost_tile_band(const uint32_t *cl, const uint32_t *cr, uint8_t *cost, int W, int Hfull, int D, int row0, int rows, int n,
                          const GuideOps &gd, cudaStream_t st);
long sweep_state_words(int W, int D);
int launch_aggregate_band(const uint8_t *guide_full, const uint32_t *cen_l_full, const uint32_t *cen_r_full, uint8_t *cost8, uint16_t *S16,
                          void *halo_ws, int W, int Hfull, int D, int row0, int rows, int n, int phases, const uint32_t *state_in,
                          uint32_t *state_out, float *dl, float *dr, const float *lut, bool plain_costs, const SgmParams &p,
                          const GuideOps &gd, uint32_t uf, cudaStream_t st);
struct StageHook { void (*fn)(void *, int); void *ctx; };   // called with VPPB200_STAGE_* when that stage has been queued
size_t sweep_halo_bytes(int W, int H, int D, int n);       // workspace of the v-sweep: inter-CTA halo lines, abort flag, P2 table
// plain_costs: the costs are plain Hamming distances (<= 24, no guided modulation): un-normalised path state in the v-sweeps
// p must satisfy sweep_params_supported(p, plain_costs)
// info_cost / info_rival: NULL, or [n][H][W] outputs of the per-pixel match info (left best / least rival cost; needs dl)
int launch_aggregate_tile(const uint8_t *img, const uint8_t *cost, uint16_t *S, void *halo_ws, int W, int H, int D, int n, float *dl,
                          float *dr, const float *lut, bool plain_costs, const SgmParams &p, const StageHook *hook, uint32_t uf,
                          cudaStream_t st, uint16_t *info_cost = nullptr, uint16_t *info_rival = nullptr);
int sweep_take_abort_flag(int *out);
int launch_s_tile_to_xyd(const uint16_t *St, uint16_t *Sx, int W, int H, int D, int n, cudaStream_t st);
void sweep_set_max_strip(int cols);
void sweep_set_enabled(int on);
void sweep_set_clusters(int c);
void vpp_set_rows_kernel(int on);
void vpp_set_md_wave(int on);
int vpp_take_md_abort_flag(int *out);
// uf: uniqueness factor (UNIQ_OFF = none); info_cost / info_rival as for launch_aggregate_tile
int launch_wta_both_subpix(const uint16_t *S, float *dl, float *dr, int W, int H, int D, const float *lut, int n, uint32_t uf,
                           cudaStream_t st, uint16_t *info_cost = nullptr, uint16_t *info_rival = nullptr);
int launch_wta_left(const uint16_t *S, float *disp, int W, int H, int D, int n, uint32_t uf, cudaStream_t st);
int launch_wta_right(const uint16_t *S, float *disp, int W, int H, int D, int n, uint32_t uf, cudaStream_t st);
int launch_subpixel(const uint16_t *S, float *disp, int W, int H, int D, int method, const float *lut, int n, cudaStream_t st);
int launch_median(const float *src, float *dst, int W, int H, int n, cudaStream_t st);
int launch_interp_clip(float *disp, int W, int H, int n, cudaStream_t st);   // _linear_interpolate(.,15,3) + clip>=0
struct TailBufs { uint8_t *u8; int *label; int *count; };       // rows of tail_stride(W) elements
static inline int tail_stride(int W) { return (W + 3) & ~3; }
int launch_tail(const float *dl, const float *dr, float *out, const RsgmDims &d, int subpixel, TailBufs tb, int n, cudaStream_t st);
// The per-pixel match info of the left view (include/vppstereo_b200.h): the same stages, each writing the part of the state it
// decides.  state / cost_out / rival_out are cropped [n][H][W]; cost_pad / rival_pad the padded maps of the fused sweep or WTA.
int launch_interp_clip_info(float *disp, const RsgmDims &d, int n, uint8_t *state, cudaStream_t st);
int launch_tail_info(const float *dl, const float *dr, float *out, const RsgmDims &d, int subpixel, TailBufs tb, int n, uint8_t *state,
                     const uint16_t *cost_pad, const uint16_t *rival_pad, uint16_t *cost_out, uint16_t *rival_out, cudaStream_t st);
const float *device_rcp_lut(cudaStream_t st);   // library-owned table for this host CPU (lazy, per device)


// t = (f * H + y) * W + x without 64-bit divisions (each costs ~100 instructions): 32-bit arithmetic whenever t fits
__device__ __forceinline__ void split_fyx(long t, int W, int H, int &x, int &y, long &f)
{
    if (t < 0x7FFFFFFFL) {
        const unsigned u = (unsigned)t, r = u / (unsigned)W, ff = r / (unsigned)H;
        x = (int)(u - r * (unsigned)W); y = (int)(r - ff * (unsigned)H); f = (long)ff;
    } else {
        x = (int)(t % W); y = (int)((t / W) % H); f = t / ((long)W * H);
    }
}
__device__ __forceinline__ int mod_w(long t, int W)
{
    return t < 0x7FFFFFFFL ? (int)((unsigned)t % (unsigned)W) : (int)(t % W);
}
}  // namespace vppb200
