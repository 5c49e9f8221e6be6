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

// ---- stage launchers (defined in the .cu files, all asynchronous on `st`) -------------------------------
int launch_pad_gray(const uint8_t *src, uint8_t *gray, const RsgmDims &d, int n, cudaStream_t st);
int launch_pad_flatbytes(const uint8_t *src, uint8_t *guide, const RsgmDims &d, int n, cudaStream_t st);
int launch_census(const uint8_t *src, uint32_t *dst, int W, int H, int n, cudaStream_t st);
void census_set_fused(int on);
int launch_census_fused(const uint8_t *src, uint32_t *dst, const RsgmDims &d, int n, cudaStream_t st);   // pad + gray + census, 1 = n/a
int launch_cost_u16(const uint32_t *cl, const uint32_t *cr, uint16_t *dsi, int W, int H, int D, int n, cudaStream_t st);
int launch_cost_u8(const uint32_t *cl, const uint32_t *cr, uint8_t *dsi, int W, int H, int D, int n, cudaStream_t st);
int launch_guided_u8(uint8_t *dsi, const float *hints, const float *valid, const RsgmDims &d, int n, cudaStream_t st);
// generic (saturating, u16 or u8 costs, any parameters) and fast (u8 costs, parameters of the sweep domain) 8-path aggregation
int launch_aggregate_generic(const uint8_t *img, const uint16_t *dsi, uint16_t *S, int W, int H, int D, int P1, int P2min,
                             float alpha, int gamma, int n, cudaStream_t st);
int launch_aggregate_generic_u8(const uint8_t *img, const uint8_t *dsi, uint16_t *S, int W, int H, int D, const SgmParams &p, int n,
                                cudaStream_t st);
int launch_aggregate_fast(const uint8_t *img, const uint8_t *dsi, uint16_t *S, int W, int H, int D, const SgmParams &p, int n,
                          cudaStream_t st);
// sgm_sweep.cu: layout-T cost volume + 4-sweep aggregation with on-chip path state (cluster per frame)
bool aggregate_tile_supported(int W, int H, int D, int n);
// do the sweeps (and the fast per-path kernels) compute these parameters exactly?  plain_costs: Hamming costs (<= 24), otherwise
// guided costs (<= 240)
bool sweep_params_supported(const SgmParams &p, bool plain_costs);
size_t tile_volume_elems(int W, int H, int D, int n);
int launch_cost_tile(const uint32_t *cl, const uint32_t *cr, uint8_t *cost, int W, int H, int D, int n, cudaStream_t st);
int launch_cost_tile_band(const uint32_t *cl, const uint32_t *cr, uint8_t *cost, int W, int Hfull, int D, int row0, int rows, int n,
                          cudaStream_t st);
long sweep_state_words(int W, int D);
int launch_aggregate_band(const uint8_t *guide_full, const uint32_t *cen_l_full, const uint32_t *cen_r_full, uint8_t *cost8, uint16_t *S16,
                          void *halo_ws, int W, int Hfull, int D, int row0, int rows, int n, int phases, const uint32_t *state_in,
                          uint32_t *state_out, float *dl, float *dr, const float *lut, bool plain_costs, const SgmParams &p,
                          cudaStream_t st);
int launch_guided_tile(uint8_t *cost, const float *hints, const float *valid, const RsgmDims &d, int n, cudaStream_t st);
struct StageHook { void (*fn)(void *, int); void *ctx; };   // called with VPPB200_STAGE_* when that stage has been queued
size_t sweep_halo_bytes(int W, int H, int D, int n);       // workspace of the v-sweep: inter-CTA halo lines, abort flag, P2 table
// plain_costs: the costs are plain Hamming distances (<= 24, no guided modulation): un-normalised path state in the v-sweeps
// p must satisfy sweep_params_supported(p, plain_costs)
int launch_aggregate_tile(const uint8_t *img, const uint8_t *cost, uint16_t *S, void *halo_ws, int W, int H, int D, int n, float *dl,
                          float *dr, const float *lut, bool plain_costs, const SgmParams &p, const StageHook *hook, cudaStream_t st);
void sweep_set_v_red(int on);
void sweep_set_v_split(int on);
int sweep_take_abort_flag(int *out);
int launch_s_tile_to_xyd(const uint16_t *St, uint16_t *Sx, int W, int H, int D, int n, cudaStream_t st);
void sweep_set_max_strip(int cols);
void sweep_set_enabled(int on);
void sweep_set_clusters(int c);
void vpp_set_rows_kernel(int on);
void vpp_set_md_wave(int on);
int vpp_take_md_abort_flag(int *out);
int launch_wta_both_subpix(const uint16_t *S, float *dl, float *dr, int W, int H, int D, const float *lut, int plane, int n,
                           cudaStream_t st);
int launch_wta_left(const uint16_t *S, float *disp, int W, int H, int D, int n, cudaStream_t st);
int launch_wta_right(const uint16_t *S, float *disp, int W, int H, int D, int n, cudaStream_t st);
int launch_subpixel(const uint16_t *S, float *disp, int W, int H, int D, int method, const float *lut, int n, cudaStream_t st);
int launch_median(const float *src, float *dst, int W, int H, int n, cudaStream_t st);
int launch_interp_clip(float *disp, int W, int H, int n, cudaStream_t st);   // _linear_interpolate(.,15,3) + clip>=0
struct TailBufs { uint8_t *u8; int *label; int *count; };       // rows of tail_stride(W) elements
static inline int tail_stride(int W) { return (W + 3) & ~3; }
int launch_tail(const float *dl, const float *dr, float *out, const RsgmDims &d, int subpixel, TailBufs tb, int n, cudaStream_t st);
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
