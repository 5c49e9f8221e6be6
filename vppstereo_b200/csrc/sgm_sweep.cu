// sgm_sweep.cu -- the 8-path SGM aggregation of compute_rsgm as FOUR sweeps with on-chip path state (sm_100a),
// bit-exact with the reference's raster recursion (RSGM/StereoSGM_SSE.hpp:13-515 via RSGM/pyrSGM.cpp:504-637;
// semantics in SURVEY.md A.4, restated per path line in sgm.cu).
//
// Why.  sgm.cu runs one launch per path (8) and every launch read-modify-writes the aggregated volume S in HBM:
// 8x the algorithmic bytes (profiles/r01_summary_v1.md).  Here S is touched once per sweep:
//   h-sweep fwd  : r0 of pass 0, one warp per image row, path state in registers, S  = L          (store)
//   v-sweep down : r1+r2+r3 of pass 0 together, S += L1+L2+L3                                      (one RMW)
//   v-sweep up   : r1+r2+r3 of pass 1 together, S += L1+L2+L3                                      (one RMW)
//   h-sweep bwd  : r0 of pass 1, S += L
//
// v-sweep (the heavy one: 6 of the 8 paths).  A TEAM of CTAs (one per SM, all resident: cooperative launch) owns one frame;
// CTA c owns a strip of 32-column groups and keeps the three paths' previous-row values L_r(x, d) of its strip in shared
// memory (~188 KB at D = 192 / 160 columns); floor(#SM / team) frames are in flight (18 at K).  LANE = COLUMN: a warp owns
// 32 adjacent columns x one third of the disparity range and walks the disparities sequentially, so L[d-1], L[d], L[d+1]
// are a register window, min_d is a running minimum, P2 is per lane -- no shuffles, no warp reductions, ~28 instructions
// per (32 pixels x 2 disparities x 3 paths).  Diagonal state is stored per LINE (ring slot = (column -/+ row) mod strip) so
// a line's state never moves; only the line that leaves the strip is handed to the neighbour CTA, through self-validating
// words in global memory (4 tag bits per word, polled: no fence, no barrier between CTAs); one __syncthreads per row.
// Lines that enter through the image border read a constant "border slot".
//
// Arithmetic: packed u16x2 DPX min/add (VIMNMX3 / VIADDMNMX) without saturation, exact inside the parameter domain that
// sweep_params_supported() states (P1, P2min, alpha, gamma are kernel arguments; P2 in [P2min, P2max], P2max = max(P2min,
// gamma); Cmax = 24 for Hamming costs, 240 for guided costs):
//   P1 <= P2min                 the recurrences form min(L[d-1], L[d+1], min + P2 - P1) + P1 in unsigned halves
//   P2max - P1 <= 255           sgm_p2_kernel packs P2 - P1 of three paths into bytes
//   Cmax + P2max <= 4095        a line handed to the neighbour CTA, relative to its part minimum, leaves the 4 tag bits of
//                               its word free; then L <= Cmax + P2max and S <= 8 * (Cmax + P2max) never saturate either
// and the v-sweeps keep their path state un-normalised only while 24 * H + P2max + 78 < 65536 (Hamming costs; see
// sgm_v2_kernel).  With the reference's effective values (7, 17, 0.25, 50) that is the fixed 24 * H + 128 rule of old.
// Parameters outside the domain are aggregated by the saturating per-path kernels of sgm.cu instead.
//
// Internal "tile" layout T of the cost volume and of S (K2 = D/2 words per pixel, G = ceil(W/32) column groups):
//   word (y, x, k) = (((y*G + x/32)*K2 + k)*32 + x%32), low half = disparity k, high half = disparity k + K2 ("split-half"
//   packing: the d-1 / d+1 neighbours of BOTH halves of word k are the halves of words k-1 / k+1, so the recurrences take
//   their neighbours as whole words -- no byte permutes in the inner loops; only the seams at d = K2-1 | K2 need one);
//   costs are uint8 (uint16 words), S is uint16 (uint32 words).  A v-sweep warp reads/writes 64 B / 128 B rows of a
//   tile; an h-sweep warp (lane = disparity chunk) gathers 8-column chunks of a tile with cp.async into a padded
//   shared-memory transpose.  vppb200 converts S to the reference's xyd order for WTA / the test tap.
#include "common.cuh"

#include <algorithm>
#include <type_traits>
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace vppb200 {

#define SW_BIG2 0x3FFF3FFFu

struct TL {
    int W, H, D, K2, G;
    long frame;        // words per frame = H*G*K2*32
};
static TL make_tl(int W, int H, int D)
{
    TL t;
    t.W = W; t.H = H; t.D = D; t.K2 = D / 2; t.G = (W + 31) / 32;
    t.frame = (long)H * t.G * t.K2 * 32;
    return t;
}

// ------------------------------------------------------------------------------------------------------------
// cost volume in layout T: popc(L ^ R[x-d]) for d <= x on rows 2..H-3, 12 elsewhere (RSGM/StereoBMHelper.cpp:29-140);
// padding columns (x >= W) hold 0.
// One warp per tile (32 columns x K2 words).  A thread owns 8 adjacent columns x one eighth of the words: the 8 left codes stay
// in registers, the right codes are two 8-word register windows (one per half of the word) that slide by one code per word
// (2 loads per 16 costs), and a word of 8 columns leaves as ONE 16-byte store (a 64-byte tile row is written by 4 lanes).  POPC (16 lanes/clk/SM) is the floor of this kernel, not the 92 MB it writes per frame.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack4(uint32_t a, uint32_t b, uint32_t c, uint32_t d)
{
    return a | (b << 8) | (c << 16) | (d << 24);
}

template <bool CHECK>
__device__ __forceinline__ void cost_pairs(const uint32_t (&L)[8], const uint32_t *__restrict__ rp, int x, int W, int K2, int k0, int k1,
                                           uint4 *__restrict__ out)
{
    // word k of column x+j holds the costs of disparities k (low byte) and k + K2 (high byte):
    // wl[j] = R[x + j - k], wh[j] = R[x + j - k - K2]; both windows slide by one code per word
    auto rload = [&](int i) -> uint32_t { return (!CHECK || (i >= 0 && i < W)) ? rp[i] : 0u; };
    uint32_t wl[8], wh[8];
#pragma unroll
    for (int j = 0; j < 8; j++) { wl[j] = rload(x + j - k0); wh[j] = rload(x + j - k0 - K2); }
#pragma unroll 4
    for (int k = k0; k < k1; k++) {
        uint32_t c[16];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            uint32_t lo = (uint32_t)__popc(L[j] ^ wl[j]), hi = (uint32_t)__popc(L[j] ^ wh[j]);
            if (CHECK) {
                if (k > x + j) lo = 12u;
                if (k + K2 > x + j) hi = 12u;
            }
            c[2 * j] = lo; c[2 * j + 1] = hi;
        }
        out[k * 4] = make_uint4(pack4(c[0], c[1], c[2], c[3]), pack4(c[4], c[5], c[6], c[7]), pack4(c[8], c[9], c[10], c[11]),
                                pack4(c[12], c[13], c[14], c[15]));
#pragma unroll
        for (int j = 7; j >= 1; j--) { wl[j] = wl[j - 1]; wh[j] = wh[j - 1]; }
        wl[0] = rload(x - k - 1);
        wh[0] = rload(x - k - 1 - K2);
    }
}

// Row bands: cl / cr / cost point at the band's first row, t.H = rows of the band, row0 / Hfull place it in the frame (the
// constant-12 rows are the first and last two rows of the FRAME).
__global__ void __launch_bounds__(256) cost_tile_kernel(const uint32_t *__restrict__ cl, const uint32_t *__restrict__ cr,
                                                        uint16_t *__restrict__ cost, TL t, long total_tiles, int row0, int Hfull,
                                                        long census_frame_stride)
{
    const long tile = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (tile >= total_tiles) return;
    const int lane = threadIdx.x & 31;
    const int xq = lane & 3, kq = lane >> 2;
    const int g = (int)(tile % t.G);
    const long row = tile / t.G;                   // row over all frames
    const int y = row0 + (int)(row % t.H);         // row inside the frame
    const long crow = (row / t.H) * census_frame_stride + (row % t.H) * (long)t.W;      // census words of this band row
    const int x = g * 32 + 8 * xq;
    const int KB = (t.K2 + 7) / 8;
    const int k0 = kq * KB, k1 = min(t.K2, k0 + KB);
    uint4 *out = reinterpret_cast<uint4 *>(cost + tile * t.K2 * 32) + xq;      // pair k of my 8 columns: out[k * 4]
    if (x >= t.W) {
        for (int k = k0; k < k1; k++) out[k * 4] = make_uint4(0, 0, 0, 0);
        return;
    }
    if (y < 2 || y >= Hfull - 2) {
        for (int k = k0; k < k1; k++) out[k * 4] = make_uint4(0x0C0C0C0Cu, 0x0C0C0C0Cu, 0x0C0C0C0Cu, 0x0C0C0C0Cu);
        return;
    }
    uint32_t L[8];
    {
        const uint4 a = *reinterpret_cast<const uint4 *>(cl + crow + x), b = *reinterpret_cast<const uint4 *>(cl + crow + x + 4);
        L[0] = a.x; L[1] = a.y; L[2] = a.z; L[3] = a.w; L[4] = b.x; L[5] = b.y; L[6] = b.z; L[7] = b.w;
    }
    const uint32_t *rp = cr + crow;
    if (g * 32 >= t.D + 2) cost_pairs<false>(L, rp, x, t.W, t.K2, k0, k1, out);       // every d <= x and every read inside the row
    else cost_pairs<true>(L, rp, x, t.W, t.K2, k0, k1, out);
}

int launch_cost_tile(const uint32_t *cl, const uint32_t *cr, uint8_t *cost, int W, int H, int D, int n, cudaStream_t st)
{
    return launch_cost_tile_band(cl, cr, cost, W, H, D, 0, H, n, st);
}
// rows [row0, row0 + rows) of frames of Hfull rows: cl / cr are the FULL census images, cost holds the band only
int launch_cost_tile_band(const uint32_t *cl, const uint32_t *cr, uint8_t *cost, int W, int Hfull, int D, int row0, int rows, int n,
                          cudaStream_t st)
{
    const TL t = make_tl(W, rows, D);
    const long tiles = (long)n * rows * t.G;
    cost_tile_kernel<<<cdiv(tiles * 32, 256), 256, 0, st>>>(cl + (long)row0 * W, cr + (long)row0 * W, reinterpret_cast<uint16_t *>(cost), t,
                                                            tiles, row0, Hfull, (long)W * Hfull);
    VPP_LAUNCH_CHECK("cost_tile_kernel");
    return VPPB200_OK;
}

// _guided_dsi (models/rsgm/rsgm.py:115-127) on the layout-T u8 volume; arithmetic as guided_u8_kernel (rsgm_ops.cu)
__global__ void guided_tile_kernel(uint8_t *__restrict__ cost, const float *__restrict__ hints, const float *__restrict__ valid,
                                   RsgmDims d, TL t, long total)
{
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int dd = (int)(i % d.D);
    const long px = i / d.D;
    const int xp = (int)(px % d.Wp), yp = (int)((px / d.Wp) % d.Hp);
    const int x = xp - d.pl, y = yp - d.pt;
    const long f = px / ((long)d.Wp * d.Hp);
    if (x < 0 || x >= d.W || y < 0 || y >= d.H) return;
    const long s = (f * d.H + y) * d.W + x;
    if (!(valid[s] > 0)) return;
    const double tt = __dsub_rn((double)hints[s], (double)dd);
    const float w = (float)__dmul_rn(10.0, __dsub_rn(1.0, exp(__ddiv_rn(-__dmul_rn(tt, tt), 2.0))));
    const long word = f * t.frame + (((long)yp * t.G + xp / 32) * t.K2 + dd % t.K2) * 32 + xp % 32;
    uint8_t *p = cost + word * 2 + (dd >= t.K2 ? 1 : 0);
    *p = (uint8_t)(uint16_t)__dmul_rn((double)*p, (double)w);
}
int launch_guided_tile(uint8_t *cost, const float *hints, const float *valid, const RsgmDims &d, int n, cudaStream_t st)
{
    const TL t = make_tl(d.Wp, d.Hp, d.D);
    long total = (long)n * d.Hp * d.Wp * d.D;
    guided_tile_kernel<<<cdiv(total, 256), 256, 0, st>>>(cost, hints, valid, d, t, total);
    VPP_LAUNCH_CHECK("guided_tile_kernel");
    return VPPB200_OK;
}

// layout-T S -> the reference's xyd order (uint16 [px][D]); one warp per tile through a padded shared-memory transpose
__global__ void __launch_bounds__(128) s_tile_to_xyd_kernel(const uint32_t *__restrict__ St, uint32_t *__restrict__ Sx, TL t,
                                                            long total_tiles)
{
    extern __shared__ uint32_t tsm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long tile = (long)blockIdx.x * 4 + warp;
    if (tile >= total_tiles) return;
    uint32_t *sm = tsm + (size_t)warp * t.K2 * 33;
    const uint32_t *src = St + tile * t.K2 * 32 + lane;
    for (int k = 0; k < t.K2; k++) sm[k * 33 + lane] = src[k * 32];
    __syncwarp();
    const int g = (int)(tile % t.G);
    const long row = tile / t.G;
    for (int c = 0; c < 32; c++) {
        const int x = g * 32 + c;
        if (x >= t.W) break;
        uint32_t *dst = Sx + (row * t.W + x) * t.K2;
        // output word m = disparities (2m, 2m+1): the low halves of words 2m, 2m+1, or (2m >= K2) the high halves of 2m-K2, 2m+1-K2
        for (int m = lane; m < t.K2; m += 32) {
            const int k = 2 * m < t.K2 ? 2 * m : 2 * m - t.K2;
            dst[m] = __byte_perm(sm[k * 33 + c], sm[(k + 1) * 33 + c], 2 * m < t.K2 ? 0x5410 : 0x7632);
        }
    }
}
int launch_s_tile_to_xyd(const uint16_t *St, uint16_t *Sx, int W, int H, int D, int n, cudaStream_t st)
{
    const TL t = make_tl(W, H, D);
    const long tiles = (long)n * H * t.G;
    const size_t smem = (size_t)4 * t.K2 * 33 * 4;
    if (smem > 48 * 1024) VPP_CUDA_TRY(cudaFuncSetAttribute(s_tile_to_xyd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    s_tile_to_xyd_kernel<<<cdiv(tiles, 4), 128, smem, st>>>(reinterpret_cast<const uint32_t *>(St),
                                                            reinterpret_cast<uint32_t *>(Sx), t, tiles);
    VPP_LAUNCH_CHECK("s_tile_to_xyd_kernel");
    return VPPB200_OK;
}

// ------------------------------------------------------------------------------------------------------------
// h-sweep: path r0 of one pass, one warp per image row, lane l owns the words [NW*l, NW*(l+1)) of a pixel, i.e. the
// disparities NW*l + j and K2 + NW*l + j (RSGM/StereoSGM_SSE.hpp:100-113,:219-236 for the recursion; the line starts with
// L = C at the pass's first column and every pixel is summed into S).  State is kept NORMALISED (L - min_d L): L_new = C +
// min(L'[d], min(L'[d-1], L'[d+1]) + P1, P2).  With the split-half packing the d-1 / d+1 neighbours of BOTH halves of word k
// are the words k-1 / k+1, so a step is two shuffles (the lanes' edge words) and, per word, VIMNMX3 + VIADDMNMX + one add;
// only the two seams (d = -1 | K2-1 below word 0, K2 | D above word K2-1) are patched with a byte permute.  Operands arrive in
// 8-column chunks: cp.async gathers the chunk's K2 rows of a tile into shared memory with odd row strides (bank-conflict-free
// transposed reads), two chunks in flight per warp; results go back through the same chunk buffer so that the global stores are
// full 32-byte sectors.
// ------------------------------------------------------------------------------------------------------------
static constexpr int HWARPS = 4;   // warps per CTA
static constexpr int HCROW = 16;   // bytes of a staged cost row: 8 columns x uint16 (16-byte pieces, dense)
#ifndef VPP_HSROW_WTA
#define VPP_HSROW_WTA 32
#endif
static constexpr int HSROW_WTA = VPP_HSROW_WTA;   // the same for the fused WTA sweep (read only)
static constexpr int HSROW = 48;   // bytes of a staged S row: 8 columns x uint32 + 16 B pad (3 pieces: odd => LDS.128 conflict-free)

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// one SGM step on normalised state: nw = c + min(w[k], min(w[k-1], w[k+1]) + P1, P2);  p2m = (P2 - P1) * 0x10001, p1x2 = P1 * 0x10001.
// FULLK: K2 == 32 * NW (every word of every lane is real); otherwise jl = index of this lane's last real word (-1: none),
// `last` = this lane holds word K2-1.
template <int NW, bool FULLK>
__device__ __forceinline__ void sw_step(const uint32_t (&w)[NW], const uint32_t (&c)[NW], uint32_t p2m, uint32_t p1x2, int lane,
                                        int lane_last, int jl, uint32_t (&nw)[NW])
{
    uint32_t ext[NW + 2];
#pragma unroll
    for (int k = 0; k < NW; k++) ext[k + 1] = w[k];
    if (FULLK) {
        // rotating shuffles: lane 0 receives word K2-1, lane 31 receives word 0 -- exactly what the two seams need
        const uint32_t up = __shfl_sync(0xFFFFFFFFu, w[NW - 1], (lane + 31) & 31);
        const uint32_t dn = __shfl_sync(0xFFFFFFFFu, w[0], (lane + 1) & 31);
        ext[0] = lane == 0 ? __byte_perm(SW_BIG2, up, 0x5410) : up;          // (BIG, L[K2-1]): below d = 0 | below d = K2
        ext[NW + 1] = lane == 31 ? __byte_perm(dn, SW_BIG2, 0x5432) : dn;    // (L[K2], BIG): above d = K2-1 | above d = D-1
    } else {
        uint32_t tail = w[0];
#pragma unroll
        for (int k = 1; k < NW; k++) if (k == jl) tail = w[k];
        const uint32_t up = __shfl_up_sync(0xFFFFFFFFu, w[NW - 1], 1);
        const uint32_t dn = __shfl_down_sync(0xFFFFFFFFu, w[0], 1);
        const uint32_t wlast = __shfl_sync(0xFFFFFFFFu, tail, lane_last);     // word K2-1
        const uint32_t w0 = __shfl_sync(0xFFFFFFFFu, w[0], 0);                // word 0
        ext[0] = lane == 0 ? __byte_perm(SW_BIG2, wlast, 0x5410) : up;
        ext[NW + 1] = dn;
        if (lane == lane_last) {
            const uint32_t seam = __byte_perm(w0, SW_BIG2, 0x5432);
#pragma unroll
            for (int k = 0; k < NW; k++) if (k == jl) ext[k + 2] = seam;
        }
    }
#pragma unroll
    for (int k = 0; k < NW; k++) {
        uint32_t t = __vimin3_u16x2(ext[k], ext[k + 2], p2m);       // min(L[d-1], L[d+1], P2 - P1)
        t = __viaddmin_u16x2(t, p1x2, w[k]);                        // min(. + P1, L[d])
        nw[k] = t + c[k];
    }
}

// min over all disparities of a warp's packed values
template <int NW>
__device__ __forceinline__ uint32_t sw_min(const uint32_t (&v)[NW])
{
    uint32_t mm = v[0];
#pragma unroll
    for (int k = 1; k < NW; k++) mm = __vminu2(mm, v[k]);
    mm = min(mm & 0xFFFFu, mm >> 16);
    return __reduce_min_sync(0xFFFFFFFFu, mm);
}

static size_t h_stage_bytes(int K2) { return (size_t)K2 * (HCROW + HSROW); }

__device__ __forceinline__ uint32_t &u4c(uint4 &v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w)); }

// MODE 0: S = L (first sweep);  MODE 1: S += L;  MODE 2: S + L is the final aggregated volume and is consumed on the
// fly by the winner-takes-all step instead of being written (RSGM/StereoBMHelper.cpp:634-750 left, :893-1015 right,
// :1072-1102 sub-pixel; same arithmetic as wta_rows_kernel in rsgm_ops.cu, which sweeps x = W-1 .. 0 like this pass).
// FULLK: K2 == NW * 32, every lane's NW words are real disparities (no validity selects)
template <int NW, int MODE, int DIR, bool FULLK>
__global__ void __launch_bounds__(HWARPS * 32) sgm_h_kernel(const uint8_t *__restrict__ img, const uint16_t *__restrict__ cost,
                                                            uint32_t *__restrict__ S, TL t, long total_rows,
                                                            float *__restrict__ disp_l, float *__restrict__ disp_r,
                                                            const float *__restrict__ lut, SgmParams prm)
{
    constexpr bool STORE = MODE == 0, WTA = MODE == 2;
    static_assert(!WTA || DIR < 0, "the fused WTA rides the backward sweep");
    extern __shared__ __align__(16) uint8_t hsm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long row = (long)blockIdx.x * HWARPS + warp;
    if (row >= total_rows) return;
    const int K2 = t.K2, W = t.W, D = t.D;
    // (MODE 2: dense 32-byte S rows -- two-way bank conflicts on the six 16-byte accesses per chunk, but five CTAs per SM instead of four)
    constexpr int SROW = MODE == 2 ? HSROW_WTA : HSROW;
    const int stage_b = K2 * (HCROW + SROW);
    uint8_t *base = hsm + (size_t)warp * 2 * stage_b;
    const uint8_t *irow = img + row * W;
    const uint16_t *crow = cost + row * (long)t.G * K2 * 32;     // tiles of this row (rows run over all frames)
    uint32_t *srow = S + row * (long)t.G * K2 * 32;
    bool wv[NW];
#pragma unroll
    for (int j = 0; j < NW; j++) wv[j] = FULLK || NW * lane + j < K2;
    const int lane_last = (K2 - 1) / NW;            // the lane that holds word K2-1 ...
    const int jl = FULLK ? NW - 1 : min(NW - 1, K2 - 1 - NW * lane);          // ... and every lane's last real word (< 0: none)
    const int nchunks = W / 8;                      // W % 16 == 0
    const int xs = DIR > 0 ? 0 : W - 1;
    const int d0 = NW * lane;                       // word j of this lane: disparities d0 + j (low half) and K2 + d0 + j (high half)

    // gather chunk q (sweep order) into stage q & 1: 16-byte pieces, one per cost row, two per S row
    auto issue = [&](int q) {
        if (q < nchunks) {
            const int xc = DIR > 0 ? q : nchunks - 1 - q;
            const int toff = ((xc >> 2) * K2) * 32 + (xc & 3) * 8;       // tile start + first column of the chunk
            uint8_t *sb = base + (q & 1) * stage_b;
            {
                const uint16_t *src = crow + toff + lane * 32;
                const uint32_t dst = smem_u32(sb) + lane * HCROW;
                for (int r0 = 0; r0 < K2; r0 += 32)
                    if (r0 + lane < K2) cp_async16(dst + r0 * HCROW, src + r0 * 32);
            }
            if (!STORE) {
                const uint32_t *src = srow + toff + (lane >> 1) * 32 + (lane & 1) * 4;
                const uint32_t dst = smem_u32(sb + K2 * HCROW) + (lane >> 1) * SROW + (lane & 1) * 16;
                for (int r0 = 0; r0 < K2; r0 += 16)
                    if (r0 + (lane >> 1) < K2) cp_async16(dst + r0 * SROW, src + r0 * 32);
            }
        }
        cp_async_commit();
    };
    issue(0);
    issue(1);

    auto p2_block = [&](int t0) -> uint32_t {
        // (P2 - P1) * 0x10001 for step t0 + lane: |I(x) - I(x - dirn)| inside the row (step 0 has no predecessor)
        const int tt = t0 + lane;
        int p2 = prm.P2min;
        if (tt > 0 && tt < W) {
            const int xx = xs + DIR * tt;
            p2 = adapt_p2(prm, irow[xx], irow[xx - DIR]);
        }
        return (uint32_t)(p2 - prm.P1) * 0x10001u;
    };
    const uint32_t p1x2 = (uint32_t)prm.P1 * 0x10001u;
    uint32_t p2v = p2_block(0), p2n = p2_block(32);
    uint32_t w[NW];
#pragma unroll
    for (int j = 0; j < NW; j++) w[j] = 0;
    // WTA right: best (cost << 16 | d) of the in-flight target pixels, a conveyor over the disparities in this lane's order:
    // ba[j] rides disparity d0 + j, bb[j] disparity K2 + d0 + j; every pixel the conveyor moves one disparity down
    uint32_t ba[NW], bb[NW];
#pragma unroll
    for (int k = 0; k < NW; k++) { ba[k] = 0xFFFFFFFFu; bb[k] = 0xFFFFFFFFu; }
    int step = 0;
    uint32_t carry = 0;
    for (int q = 0; q < nchunks; q++) {
        cp_async_wait<1>();
        __syncwarp();
        uint8_t *sb = base + (q & 1) * stage_b;
        uint8_t *ssb = sb + K2 * HCROW;
        const int xlo = (DIR > 0 ? q : nchunks - 1 - q) * 8;
        // this lane's rows of the chunk: 8 pixels x NW words, costs (uint16) and S words
        uint4 cv[NW], s0[NW], s1[NW];
#pragma unroll
        for (int j = 0; j < NW; j++) {
            cv[j] = make_uint4(0, 0, 0, 0); s0[j] = cv[j]; s1[j] = cv[j];
            if (wv[j]) {
                cv[j] = *reinterpret_cast<const uint4 *>(sb + (NW * lane + j) * HCROW);
                if (!STORE) {
                    s0[j] = *reinterpret_cast<const uint4 *>(ssb + (NW * lane + j) * SROW);
                    s1[j] = *reinterpret_cast<const uint4 *>(ssb + (NW * lane + j) * SROW + 16);
                }
            }
        }

        // WTA: the chunk's 8 left minima (cost << 16 | d) and 8 retired right winners are parked in shared memory (uniform values,
        // one store each); the sub-pixel step is deferred to the end of the chunk, where the final S of all 8 pixels sits in the
        // stage buffer and lanes 0..7 finish one pixel each
        uint32_t *wout = reinterpret_cast<uint32_t *>(hsm + (size_t)HWARPS * 2 * stage_b) + warp * 16;
        const bool nomask = xlo >= D - 1;             // every d <= x in this chunk: the left arg-min needs no range mask
#pragma unroll
        for (int pp = 0; pp < 8; pp++, step++) {
            const int p = DIR > 0 ? pp : 7 - pp;
            if ((step & 31) == 0 && step > 0) { p2v = p2n; p2n = p2_block(step + 32); }
            const uint32_t bsel = (p & 1) ? 0x4342 : 0x4140;                                   // two uint8 -> u16x2
            uint32_t cc[NW];
#pragma unroll
            for (int j = 0; j < NW; j++) cc[j] = __byte_perm(u4c(cv[j], p >> 1), 0, bsel);
            const uint32_t p2m = __shfl_sync(0xFFFFFFFFu, p2v, step & 31);
            uint32_t nw[NW];
            if (step == 0) {
#pragma unroll
                for (int j = 0; j < NW; j++) nw[j] = cc[j];
            } else {
                sw_step<NW, FULLK>(w, cc, p2m, p1x2, lane, lane_last, jl, nw);
            }
#pragma unroll
            for (int j = 0; j < NW; j++) if (!wv[j]) nw[j] = SW_BIG2;
            const uint32_t m2 = sw_min<NW>(nw) * 0x10001u;
            uint32_t fin[NW];
#pragma unroll
            for (int j = 0; j < NW; j++) {
                w[j] = nw[j] - m2;
                uint32_t &acc = p < 4 ? u4c(s0[j], p) : u4c(s1[j], p - 4);
                acc = STORE ? nw[j] : acc + nw[j];
                fin[j] = acc;
            }
            if (WTA) {
                const int x = xlo + p;
                uint32_t ka[NW], kb[NW];              // (cost << 16 | d) of the low-half and of the high-half disparities
#pragma unroll
                for (int j = 0; j < NW; j++) {
                    // (multiply-add and one logic op: the byte-permute unit shares the integer pipe this kernel is bound by)
                    ka[j] = wv[j] ? fin[j] * 65536u + (uint32_t)(d0 + j) : 0xFFFFFFFFu;
                    kb[j] = wv[j] ? ((fin[j] & 0xFFFF0000u) | (uint32_t)(K2 + d0 + j)) : 0xFFFFFFFFu;
                }
                // left: first arg-min over d <= min(D-1, x)
                const int end = min(D - 1, x);
                uint32_t m = 0xFFFFFFFFu;
                if (nomask) {
#pragma unroll
                    for (int k = 0; k < NW; k++) m = min(m, min(ka[k], kb[k]));
                } else {
#pragma unroll
                    for (int k = 0; k < NW; k++) {
                        m = min(m, (d0 + k <= end) ? ka[k] : 0xFFFFFFFFu);
                        m = min(m, (K2 + d0 + k <= end) ? kb[k] : 0xFFFFFFFFu);
                    }
                }
                m = __reduce_min_sync(0xFFFFFFFFu, m);
                wout[p] = m;
                // right: every in-flight target absorbs its disparity slot, slot d = 0 retires to disp_r[x], the conveyor moves
                // one disparity down: within the halves by register moves, between lanes by a rotating shuffle (lane 31
                // receives lane 0's slots: its low-half tail takes d = K2 from there, its high-half tail starts empty)
#pragma unroll
                for (int k = 0; k < NW; k++) { ba[k] = min(ba[k], ka[k]); bb[k] = min(bb[k], kb[k]); }
                if (lane == 0) wout[8 + p] = ba[0];
                const uint32_t fa = __shfl_sync(0xFFFFFFFFu, ba[0], (lane + 1) & 31);
                const uint32_t fb = __shfl_sync(0xFFFFFFFFu, bb[0], (lane + 1) & 31);
#pragma unroll
                for (int k = 0; k < NW - 1; k++) { ba[k] = ba[k + 1]; bb[k] = bb[k + 1]; }
                if (FULLK) {
                    ba[NW - 1] = lane == 31 ? fb : fa;
                    bb[NW - 1] = lane == 31 ? 0xFFFFFFFFu : fb;
                } else {
                    // the lane that holds word K2-1: its low-half tail (disparity K2-1) takes over disparity K2 = lane 0's first
                    // high-half slot; slots past K2-1 stay empty
                    const uint32_t fb0 = __shfl_sync(0xFFFFFFFFu, fb, 31);          // = lane 0's bb[0] before the move
                    ba[NW - 1] = fa; bb[NW - 1] = fb;
                    if (lane >= lane_last) {
#pragma unroll
                        for (int k = 0; k < NW; k++) {
                            if (lane > lane_last || k > jl) { ba[k] = 0xFFFFFFFFu; bb[k] = 0xFFFFFFFFu; }
                            else if (k == jl) { ba[k] = fb0; bb[k] = 0xFFFFFFFFu; }
                        }
                    }
                }
            }
        }
        if (WTA) {
            // final S of the chunk's 8 pixels -> the (consumed) S rows of the stage; disparity d of pixel p sits in half d / K2 of
            // column p of row d % K2
#pragma unroll
            for (int j = 0; j < NW; j++) {
                if (wv[j]) {
                    *reinterpret_cast<uint4 *>(ssb + (NW * lane + j) * SROW) = s0[j];
                    *reinterpret_cast<uint4 *>(ssb + (NW * lane + j) * SROW + 16) = s1[j];
                }
            }
            __syncwarp();
            if (lane < 8) {
                const int x = xlo + lane;
                const uint32_t m = wout[lane];
                const int best = (int)(m & 0xFFFFu);
                float o = (float)best;
                if (x >= 1 && x <= W - 2) {
                    if (best > 0) {
                        auto at = [&](int d) -> int {
                            return *reinterpret_cast<const uint16_t *>(ssb + (d < K2 ? d : d - K2) * SROW + lane * 4 + (d < K2 ? 0 : 2));
                        };
                        const int c0 = at(best - 1), c1 = (int)(m >> 16);
                        // best = D-1 reads the next pixel's d = 0 (xyd stream order): column x+1, in the previous chunk for lane 7
                        const int c2 = best + 1 < D ? at(best + 1)
                                                    : (lane < 7 ? (int)*reinterpret_cast<const uint16_t *>(ssb + (lane + 1) * 4) : (int)carry);
                        const int lower = min(c1 - c0, c1 - c2);            // <= 0
                        o = __fadd_rn((float)best, __fmul_rn((float)(c2 - c0), lut[-lower]));
                    } else {
                        o = -10.0f;
                    }
                }
                disp_l[row * W + x] = o;
                disp_r[row * W + x] = (float)(wout[8 + lane] & 0xFFFFu);
            }
            carry = __shfl_sync(0xFFFFFFFFu, s0[0].x, 0) & 0xFFFFu;         // S(d = 0) of the chunk's first column
        } else {
#pragma unroll
            for (int j = 0; j < NW; j++) {
                if (wv[j]) {
                    *reinterpret_cast<uint4 *>(ssb + (NW * lane + j) * SROW) = s0[j];
                    *reinterpret_cast<uint4 *>(ssb + (NW * lane + j) * SROW + 16) = s1[j];
                }
            }
            __syncwarp();
            // write the chunk's S rows back: two 16-byte pieces = one 32-byte sector per row
            const int toff = ((xlo >> 5) * K2) * 32 + (xlo & 31);
            uint32_t *dst = srow + toff + (lane >> 1) * 32 + (lane & 1) * 4;
            const uint8_t *src = ssb + (lane >> 1) * SROW + (lane & 1) * 16;
            for (int r0 = 0; r0 < K2; r0 += 16)
                if (r0 + (lane >> 1) < K2)
                    *reinterpret_cast<uint4 *>(dst + r0 * 32) = *reinterpret_cast<const uint4 *>(src + r0 * SROW);
        }
        __syncwarp();
        issue(q + 2);
    }
    cp_async_wait<0>();
}

template <int NW, int MODE, int DIR>
static int run_h_t(const uint8_t *img, const uint16_t *cost, uint32_t *S, const TL &t, int n, float *dl, float *dr,
                   const float *lut, const SgmParams &prm, cudaStream_t st)
{
    const long rows = (long)n * t.H;
    const int blocks = cdiv(rows, HWARPS);
    const size_t stage = MODE == 2 ? (size_t)t.K2 * (HCROW + HSROW_WTA) : h_stage_bytes(t.K2);
    const size_t smem = (size_t)HWARPS * 2 * stage + (MODE == 2 ? (size_t)HWARPS * 16 * 4 : 0);
    auto kern = t.K2 == NW * 32 ? sgm_h_kernel<NW, MODE, DIR, true> : sgm_h_kernel<NW, MODE, DIR, false>;
    if (smem > 48 * 1024) VPP_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<blocks, HWARPS * 32, smem, st>>>(img, cost, S, t, rows, dl, dr, lut, prm);
    VPP_LAUNCH_CHECK("sgm_h_kernel");
    return VPPB200_OK;
}

// mode 0: forward sweep, S = L;  mode 1: backward sweep, S += L;  mode 2: backward sweep fused with WTA (dl, dr, lut)
static int run_h(const uint8_t *img, const uint16_t *cost, uint32_t *S, const TL &t, int mode, int n, float *dl, float *dr,
                 const float *lut, const SgmParams &prm, cudaStream_t st)
{
#define VPP_RUN_H(NW)                                                                                                  \
    return mode == 0 ? run_h_t<NW, 0, 1>(img, cost, S, t, n, nullptr, nullptr, nullptr, prm, st)                       \
         : mode == 1 ? run_h_t<NW, 1, -1>(img, cost, S, t, n, nullptr, nullptr, nullptr, prm, st)                      \
                     : run_h_t<NW, 2, -1>(img, cost, S, t, n, dl, dr, lut, prm, st)
    switch ((t.K2 + 31) / 32) {
        case 1: VPP_RUN_H(1);
        case 2: VPP_RUN_H(2);
        case 3: VPP_RUN_H(3);
        default: VPP_RUN_H(4);
    }
#undef VPP_RUN_H
}

// ------------------------------------------------------------------------------------------------------------
// v-sweep: paths r1, r2, r3 of one pass, a team of CTAs per frame, lane = column, path state in shared memory
// ------------------------------------------------------------------------------------------------------------
struct VArgs {
    TL t;
    int n;
    int pass;          // 0: top-down (di = dj = +1), 1: bottom-up (di = dj = -1)
    int csize;         // CTAs per team (one frame)
    int GC;            // 32-column groups per CTA, ceil(G / csize)
    uint32_t p1x2;     // P1 * 0x10001
    // Row bands (a frame split over several GPUs, SURVEY.md 8e row 5): t.H is the band's row count, the volumes hold the band's
    // rows only.  pass_start = the band begins with the pass's first image row (L = C there); otherwise the sweep continues from
    // `state_in`, the path state of the row before the band as another band's sweep left it in `state_out`:
    // [frame][3 paths][G*32 columns][K2 words], then [frame][3][G*32][VPARTS] part minima (state_words per frame in total).
    int pass_start;
    const uint32_t *state_in;
    uint32_t *state_out;
    long state_words;
};

#ifndef VPP_VREGS
#define VPP_VREGS 96
#endif
#ifndef VPP_VPARTS
#define VPP_VPARTS 3
#endif
#ifndef VPP_VU
#define VPP_VU 8
#endif
static constexpr int VPARTS = VPP_VPARTS;   // warps per column group (each owns a share of the disparity pairs)
static constexpr int VU = VPP_VU;           // disparity pairs per operand block (software pipelined)

__device__ __forceinline__ uint32_t add3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r;
    asm("{\n\t.reg .u32 t;\n\tadd.u32 t, %1, %2;\n\tadd.u32 %0, t, %3;\n\t}" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---- halo exchange between the CTAs of a team (the CTAs that share one frame): self-validating words in global
// memory.  Handed-over state words are < 2^28 (two uint16 values <= Cmax + P2max <= 4095 once taken relative to their line's
// part minimum: sweep_params_supported), so the
// top four bits carry a tag that changes with the row; the consumer polls a word until its tag is the expected one.  No
// fence, no barrier between CTAs: every word is its own flag (relaxed gpu-scope stores and loads go through L2).
__device__ __forceinline__ void st_relaxed_gpu(uint32_t *p, uint32_t v)
{
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_gpu(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
static constexpr uint32_t HALO_INVALID = 0xF0000000u;

// ------------------------------------------------------------------------------------------------------------
// v-sweep, second generation.  Mapping as in the first generation (git history: sgm_v_kernel; team of CTAs per frame, lane =
// column, a warp owns 32 columns x one third of the disparity pairs, per-line ring slots in shared memory), rebuilt around what
// its profile showed (profiles/r01_summary_v4.md: 57 % issue utilisation, barrier the largest stall, 392 of 1352
// instructions per warp and row outside the disparity loop):
//  * NO CTA-wide barrier per row.  With per-line ring slots the only true dependencies of (column group g, row t) are the rows
//    t-1 of groups g-1, g, g+1 (one diagonal line crosses each group boundary).  Every warp signals "row done" on an mbarrier
//    of its group (arrive) and waits on the three it depends on (try_wait: suspended in hardware, no polling instructions);
//    groups drift up to one row apart, the tail of a row overlaps the head of the next one, and the edge groups (whose lines
//    the neighbour CTAs wait for) run ahead.
//    The ring phase runs on across frames, so the frame boundary needs no barrier either.
//  * The line that enters from the neighbour CTA is deposited straight into the ring slot its predecessor line just left
//    (the slot is free exactly then), so every lane reads its own ring slot: no halo slots, no select in the loop, no
//    shared-memory bank conflicts.
//  * L is kept WITHOUT subtracting the predecessor's minimum per path (NORM = false): with Lt = L + (running sum of the minima)
//    the recurrence is Lt = C + min(Lt[d], Lt[d+-1] + P1, min Lt + P2) and the reference's value is Lt - min_prev, so the three
//    subtractions per disparity pair collapse into ONE constant per pixel folded into the S update:
//    S += Lt1 + Lt2 + Lt3 - (m1 + m2 + m3).  The minimum grows by at most max(C) per row, so Lt <= 24 * H + P2max: the state
//    stays un-normalised while 24 * H + P2max + 78 < 65536 for Hamming costs (H <= 2700 with the default P2max = 50);
//    guided costs (<= 240) take NORM = true.  Lines handed to a neighbour CTA travel normalised by their own part minimum
//    (<= Cmax + P2max per half word), which keeps the 4 tag bits of the self-validating words free.
//  * P2 of the three paths comes from a per-pixel table (sgm_p2_kernel: one word instead of four image loads and three
//    float evaluations per warp and row, and the flat-stream wrap rules live in one place).
//  * a timed-out halo wait raises a flag in global memory (checked by the host) and lets the grid run to completion with
//    undefined results, instead of trapping the context.
// ------------------------------------------------------------------------------------------------------------
#define SW_INF2 0xFFFFFFFFu

// (P2 - P1) of the three paths of one pass for every pixel, packed q1 | q2 << 8 | q3 << 16; [n][H][G*32] words.
// P2 = adaptP2(I(p), I(p - r)) with I read from the FLAT byte stream of the guide (RSGM/StereoSGM.hpp:92-99,
// StereoSGM_SSE.hpp:221,:238-243: on the row after the pass's first row the "previous line" is that same row).
// Row bands: the table covers rows [row0, row0 + Hb) of frames of H rows (img_all = the full guide images).
// One thread = 4 adjacent pixels of a row (one 16-byte store); grid.y = frame * Hb + band row.
__global__ void __launch_bounds__(256) sgm_p2_kernel(const uint8_t *__restrict__ img_all, uint32_t *__restrict__ p2q, int W, int H,
                                                     int G32, int pass, int row0, int Hb, SgmParams prm)
{
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (x0 >= G32) return;
    const long r = blockIdx.y;                            // f * Hb + band row
    const int i = row0 + (int)(r % Hb);
    const long f = r / Hb;
    const int dj = pass == 0 ? 1 : -1, di = dj, i1 = pass == 0 ? 0 : H - 1;
    uint4 out = make_uint4(0u, 0u, 0u, 0u);
    if (i != i1) {
        const int npx = W * H;                            // (a frame's tile volume fits 31 bits, so does its pixel count)
        const uint8_t *img = img_all + f * (long)npx;
        const int s = (i - i1) * di;
        const int il = s == 1 ? i : i - di;
        const uint8_t *rc = img + i * W, *rl = img + il * W;
        const int lbase = il * W;
        uint32_t o[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int xr = min(x0 + u, W - 1);
            int q1 = lbase + xr - dj, q3 = lbase + xr + dj;
            q1 = q1 < 0 ? 0 : (q1 >= npx ? npx - 1 : q1);
            q3 = q3 < 0 ? 0 : (q3 >= npx ? npx - 1 : q3);
            const int ipc = rc[xr], ip1 = img[q1], ip2 = rl[xr], ip3 = img[q3];
            o[u] = (uint32_t)(adapt_p2(prm, ipc, ip1) - prm.P1) | ((uint32_t)(adapt_p2(prm, ipc, ip2) - prm.P1) << 8) |
                   ((uint32_t)(adapt_p2(prm, ipc, ip3) - prm.P1) << 16);
        }
        out = make_uint4(o[0], o[1], o[2], o[3]);
    }
    *reinterpret_cast<uint4 *>(p2q + r * G32 + x0) = out;
}

// Raised by a hand-off wait that timed out (a CTA of the team not resident / not progressing: the protocol needs all CTAs of the
// cooperative grid on the device at once).  The grid then runs to completion with undefined results instead of trapping the
// context; the host reads the flag with vppb200_async_error().
__device__ unsigned int g_sweep_abort = 0;

// bounded wait on a tagged halo word; on a timeout the abort flag is raised and every later wait returns at once
__device__ __noinline__ uint32_t halo_wait2(const uint32_t *p, uint32_t tag, uint32_t *abort_flag)
{
    for (uint32_t spin = 0; spin < (1u << 25); spin++) {
        const uint32_t v = ld_relaxed_gpu(p);
        if ((v >> 28) == tag) return v & 0x0FFFFFFFu;
        if ((spin & 1023u) == 1023u && ld_relaxed_gpu(abort_flag) != 0u) return 0u;
    }
    st_relaxed_gpu(abort_flag, 1u);
    return 0u;
}

#ifdef VPP_TRACE
// debug build only (tools/vtrace.py): clock64 stamps of one CTA's warps over a window of rows
static constexpr int TR_ROW0 = 100, TR_ROWS = 24, TR_STAMPS = 12, TR_CTA = 3;
__device__ unsigned long long g_vtrace[32 * TR_ROWS * TR_STAMPS];
#define VTRACE(k)                                                                                                      \
    do {                                                                                                               \
        if (blockIdx.x == TR_CTA && lane == 0 && t >= TR_ROW0 && t < TR_ROW0 + TR_ROWS)                                 \
            g_vtrace[(warp * TR_ROWS + (t - TR_ROW0)) * TR_STAMPS + (k)] = clock64();                                  \
    } while (0)
#else
#define VTRACE(k) do { } while (0)
#endif

struct VPath2 {
    uint32_t cur;      // word k of the predecessor: Lt[k], Lt[k + K2]
    uint32_t prev;     // word k-1 (for word 0: the seam (inf, Lt[K2-1]))
    uint32_t q;        // (min + P2 - P1) x2
    uint32_t ng;       // NORM: min of the predecessor
    uint32_t mr;       // running min of the new values
};

__device__ __forceinline__ void red_add_u32(uint32_t *p, uint32_t v)
{
    asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// One block of up to VU words for the three paths.  s* = predecessor state rows of the block (stride NS), w* = this row's state
// rows (same slots), Sg = the block's S words (stride 32).  GUARD: only the first `cnt` words exist; `last`: the block ends this
// warp's share, whose upper neighbour word was read before the column group's barrier (wr*).
// RED: S += goes out as a fire-and-forget reduction to L2 (the addend's halves are <= 3 * (Cmax + P2max) and S's halves never
// overflow, so the 32-bit add is exact for both halves): no load of S, no operand registers, no latency to hide
template <int NS, bool GUARD, bool NORM, bool RED>
__device__ __forceinline__ void v2_block(const uint32_t (&cb)[VU], const uint32_t (&sb)[VU], const uint32_t *s1,
                                         const uint32_t *s2, const uint32_t *s3, uint32_t *w1, uint32_t *w2, uint32_t *w3,
                                         uint32_t wr1, uint32_t wr2, uint32_t wr3, VPath2 &p1, VPath2 &p2, VPath2 &p3,
                                         uint32_t negm, uint32_t p1x2, uint32_t *Sg, int cnt, bool last)
{
    uint32_t nx1[VU], nx2[VU], nx3[VU];
    uint32_t tp1 = 0, tp2 = 0, tp3 = 0;
#pragma unroll
    for (int u = 0; u < VU; u++) {
        if (u + 1 < VU) {
            if (!GUARD || u + 1 < cnt) { nx1[u] = s1[(u + 1) * NS]; nx2[u] = s2[(u + 1) * NS]; nx3[u] = s3[(u + 1) * NS]; }
            else { nx1[u] = wr1; nx2[u] = wr2; nx3[u] = wr3; }
        } else {
            if (last) { nx1[u] = wr1; nx2[u] = wr2; nx3[u] = wr3; }
            else { nx1[u] = s1[VU * NS]; nx2[u] = s2[VU * NS]; nx3[u] = s3[VU * NS]; }
        }
    }
#pragma unroll
    for (int u = 0; u < VU; u++) {
        if (!GUARD || u < cnt) {
            const uint32_t c = __byte_perm(cb[u], 0, 0x4140);                        // two uint8 costs -> u16x2
            // split-half packing: the neighbours d-1 / d+1 of both halves are the words k-1 / k+1 as they stand
            uint32_t t1 = __vimin3_u16x2(p1.prev, nx1[u], p1.q), t2 = __vimin3_u16x2(p2.prev, nx2[u], p2.q),
                     t3 = __vimin3_u16x2(p3.prev, nx3[u], p3.q);                     // min(Lt[d-1], Lt[d+1], min + P2 - P1)
            t1 = __viaddmin_u16x2(t1, p1x2, p1.cur);                                 // min(. + P1, Lt[d])
            t2 = __viaddmin_u16x2(t2, p1x2, p2.cur);
            t3 = __viaddmin_u16x2(t3, p1x2, p3.cur);
            uint32_t sum;
            if (NORM) {
                t1 = (t1 + c) + p1.ng * 0xFFFEFFFFu; t2 = (t2 + c) + p2.ng * 0xFFFEFFFFu; t3 = (t3 + c) + p3.ng * 0xFFFEFFFFu;
                sum = (t1 + t2) + t3;
            } else {
                // packed halves may carry into each other inside the sum; the final halves (<= 3 * (Cmax + P2max)) are exact mod 2^32
                t1 += c; t2 += c; t3 += c;
                sum = add3(t1, t2, t3) + negm;
            }
            w1[u * NS] = t1; w2[u * NS] = t2; w3[u * NS] = t3;
            if (u & 1) {
                p1.mr = __vimin3_u16x2(p1.mr, tp1, t1); p2.mr = __vimin3_u16x2(p2.mr, tp2, t2); p3.mr = __vimin3_u16x2(p3.mr, tp3, t3);
            } else if (GUARD && u + 1 >= cnt) {
                p1.mr = __vminu2(p1.mr, t1); p2.mr = __vminu2(p2.mr, t2); p3.mr = __vminu2(p3.mr, t3);
            }
            tp1 = t1; tp2 = t2; tp3 = t3;
            if (RED) red_add_u32(Sg + u * 32, sum);
            else Sg[u * 32] = sum + sb[u];
            p1.prev = p1.cur; p2.prev = p2.cur; p3.prev = p3.cur;
            p1.cur = nx1[u]; p2.cur = nx2[u]; p3.cur = nx3[u];
        }
    }
}

// NS = GC * 32 ring slots + the border slot.
// FULL: every warp's share of the words is a whole number of VU-blocks (no guards in the inner loop).  NORM, RED: see above.
// halo: [CTA][r1 | r3][row parity][K2 state words + VPARTS part minima] inbound buffers, then one abort word at the end
// Register cap: 96 where the S update is a reduction (no operand registers for S; no spills): the one-CTA-per-SM grid then
// leaves a quarter of the register file and ~30 KB of shared memory per SM to the front / tail kernels of the neighbouring
// batches, which run beside the sweep (measured: the sweep alone 6.09 -> 6.39 ms, the pipelined step 23.7 -> 23.3 ms)
// BAND: the launch covers a row band of taller frames (state import / export at the band's ends); whole-frame launches are
// compiled without that code (it costs the hot loop 0.3 ms per launch under the register cap).  Band launches take the 128 cap
// (a band's sweep does not share the SMs with the phases of neighbouring batches; under 96 registers the runtime P1 made the
// band kernels spill).  The residency plan (v_resident_ctas) is computed for 128 registers either way.
template <int NS, bool FULL, bool NORM, bool RED, bool BAND>
__global__ void __maxnreg__(RED && !BAND ? VPP_VREGS : 128) sgm_v2_kernel(const uint32_t *__restrict__ p2q_all,
                                                                                 const uint16_t *__restrict__ cost_all,
                                                                                 uint32_t *__restrict__ S_all, uint32_t *halo,
                                                                                 uint32_t *abort_flag, VArgs a)
{
    extern __shared__ __align__(16) uint32_t smem[];
    using SW = uint32_t;
    const int rank = (int)(blockIdx.x % a.csize);
    const int cid = blockIdx.x / a.csize, nteams = gridDim.x / a.csize;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int W = a.t.W, H = a.t.H, K2 = a.t.K2, G = a.t.G;
    const uint32_t p1x2 = a.p1x2;
    constexpr int BIGS = NS - 1;
    const int part = warp % VPARTS;
    const int g_first = rank * a.GC;
    const int ng = min(a.GC, G - g_first);
    // edge groups on the highest warp ids (the schedulers prefer them): their lines are what the neighbour CTAs wait for
    int gl;
    {
        const int wq = warp / VPARTS, nG = a.GC;
        if (wq == nG - 1) gl = ng - 1;
        else if (wq == nG - 2) gl = ng >= 2 ? 0 : nG;
        else gl = (wq + 1 < ng - 1) ? wq + 1 : nG;
    }
    const int n = ng * 32;
    const int x0 = g_first * 32;
    const int dj = a.pass == 0 ? 1 : -1, di = dj;
    const int i1 = a.pass == 0 ? 0 : H - 1;
    const int KP = (K2 + VPARTS - 1) / VPARTS;
    const int k0 = part * KP, k1 = min(K2, k0 + KP);
    const bool active = gl < ng && k0 < k1;
    const int nact = (K2 + KP - 1) / KP;

    uint32_t *st = smem;                            // [3][K2][NS]   Lt of the previous row, per line
    uint32_t *mn = st + 3 * K2 * NS;                // [3][VPARTS][NS] min_d of each share of that row
    for (int idx = tid; idx < 3 * K2 * NS; idx += blockDim.x) st[idx] = SW_INF2;
    for (int idx = tid; idx < 3 * VPARTS * NS; idx += blockDim.x) mn[idx] = (idx % NS == BIGS) ? 0u : 0xFFFFu;
    // [GC][2] "row done" mbarriers behind the minima (8-byte aligned), expected arrivals = warps per group
    uint64_t *mbar = reinterpret_cast<uint64_t *>(smem + ((3 * K2 * NS + 3 * VPARTS * NS + 3) & ~3));
    if (tid < 2 * a.GC) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(mbar + tid)), "r"(nact) : "memory");
    const int HL = K2 + VPARTS;
    const bool has1 = rank + dj >= 0 && rank + dj < a.csize, has3 = rank - dj >= 0 && rank - dj < a.csize;
    uint32_t *in1 = halo + ((size_t)blockIdx.x * 2 + 0) * 2 * HL, *in3 = halo + ((size_t)blockIdx.x * 2 + 1) * 2 * HL;
    uint32_t *push1 = halo + ((size_t)(blockIdx.x + dj) * 2 + 0) * 2 * HL;       // neighbour's inbound r1 (valid if has1)
    uint32_t *push3 = halo + ((size_t)(blockIdx.x - dj) * 2 + 1) * 2 * HL;       // neighbour's inbound r3 (valid if has3)
    const int gl_leave1 = dj > 0 ? ng - 1 : 0, lane_leave1 = dj > 0 ? 31 : 0;
    const int gl_leave3 = dj > 0 ? 0 : ng - 1, lane_leave3 = dj > 0 ? 0 : 31;
    // an r1 line enters where r3 lines leave (from rank - dj) and vice versa
    const bool enter1 = has3 && gl == gl_leave3, enter3 = has1 && gl == gl_leave1;
    for (int idx = tid; idx < 2 * HL; idx += blockDim.x) { st_relaxed_gpu(in1 + idx, HALO_INVALID); st_relaxed_gpu(in3 + idx, HALO_INVALID); }
    __threadfence();
    cg::this_grid().sync();                         // every inbound buffer is invalidated before anybody pushes
    if (!active) return;                            // no CTA-wide barrier below this line

    const int lc = gl * 32 + lane;
    const int x = x0 + lc;
    const int g = g_first + gl;
    const int G32 = G * 32;
    const bool border1 = (x - dj < 0) || (x - dj >= W), border3 = (x + dj < 0) || (x + dj >= W);
    // "Row done" hand-shake between column groups: one mbarrier per (group, row parity) in shared memory, expected count = the
    // group's warps.  A warp ARRIVES (release) when its row t is complete; before row t+1 a warp WAITS (acquire; try_wait
    // suspends the warp in hardware, a waiting warp costs no issue slots) on the barriers of its own group and of its two
    // neighbours ON THE RING of the strip's groups -- the first and the last group are neighbours too: the ring slot a line
    // leaves on one side is taken by the line that enters (or starts at the image border) on the other side in the very next
    // row.  Waiting does not count as arriving, so there is no cyclic wait.  Two barriers per group: a group may finish row t+1
    // before a neighbour has looked at its row t (but never row t+2), so the phase parity a waiter names is unambiguous.
    const int g_prev = gl == 0 ? ng - 1 : gl - 1, g_next = gl == ng - 1 ? 0 : gl + 1;
    const uint32_t mb_base = smem_u32(mbar);
    const unsigned group_threads = (unsigned)nact * 32u;
    auto group_barrier = [&]() {                     // rendezvous of the group's own warps inside a row
        if (nact > 1) asm volatile("bar.sync %0, %1;" ::"r"(1 + gl), "r"(group_threads) : "memory");
        else __syncwarp();
    };
    auto row_done = [&](unsigned tt) {               // this warp's row tt is complete (state, minima, outbound lines written)
        __syncwarp();
        if (lane == 0)
            asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(mb_base + (uint32_t)(2 * gl + (int)(tt & 1u)) * 8u)
                         : "memory");
    };
    auto try_row = [&](int gq, unsigned tt) -> uint32_t {
        const uint32_t addr = mb_base + (uint32_t)(2 * gq + (int)(tt & 1u)) * 8u, parity = (tt >> 1) & 1u;
        uint32_t ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
        return ok;
    };
    // (Measured alternatives, all slower than this loop's 6.11 ms per launch: three blocking try_waits one after the other 6.43 ms;
    // one barrier per group that collects the arrivals of all the warps the group depends on, polled alone, 6.34 ms with
    // try_wait, 6.48 ms with test_wait, 6.41-6.9 ms with test_wait + nanosleep 30 / 100 / 300.  A suspend-time hint on the try_wait (2 us, 10 ms)
    // takes the polling instructions away but not the wait: 6.20 vs 6.09 ms, same step time.  Here a try_wait on a phase
    // that is already complete returns at once, so the loop polls the pending ones ~20 times per row: fast wake-up without a
    // tight spin that would starve the lower-priority working warps.)
    auto wait_rows = [&](unsigned tt) {              // every warp of this group and of its ring neighbours has completed row tt
        uint32_t a0 = 0, a1 = 0, a2 = 0;             // the three waits are issued back to back
        do {
            if (!a0) a0 = try_row(g_prev, tt);
            if (!a1) a1 = try_row(g_next, tt);
            if (!a2) a2 = try_row(gl, tt);
        } while (!(a0 & a1 & a2));
    };

    unsigned t = 0;                                 // rows processed by this team so far, over all its frames
    int sh = 0;                                     // t mod n: the ring phase runs on across frames
    uint32_t cb[VU], sb[VU];
#pragma unroll
    for (int u = 0; u < VU; u++) { cb[u] = 0; sb[u] = 0; }
    uint32_t p2w = 0;                               // packed (P2 - P1) of the three paths for the coming row
    for (int f = cid; f < a.n; f += nteams) {
        const uint16_t *cost_f = cost_all + f * a.t.frame + lane;
        SW *S_f = reinterpret_cast<SW *>(S_all) + f * a.t.frame + lane;
        const uint32_t *p2_f = p2q_all + (long)f * H * G32 + x;
        auto load_block = [&](const uint16_t *cp, const SW *sp, int cnt, uint32_t (&c)[VU], uint32_t (&sv)[VU], bool with_s) {
#pragma unroll
            for (int u = 0; u < VU; u++) {
                if (FULL || u < cnt) {
                    c[u] = cp[u * 32];
                    sv[u] = (!RED && with_s) ? sp[u * 32] : 0u;
                }
            }
        };
        const bool cont = BAND && !a.pass_start;    // row band that continues a sweep: its first row is an ordinary row
        if (f == cid) load_block(cost_f + (((long)i1 * G + g) * K2 + k0) * 32, S_f + (((long)i1 * G + g) * K2 + k0) * 32, k1 - k0, cb, sb, cont);
        for (int s = 0; s < H; s++, t++) {
            const int i = i1 + s * di;
            // ring slots: a line moving +1 column per row sits in slot (lc - t) mod n, one moving -1 in (lc + t) mod n
            int slotA = lc - sh; if (slotA < 0) slotA += n;
            int slotB = lc + sh; if (slotB >= n) slotB -= n;
            const int d1 = dj > 0 ? slotA : slotB, d2 = lc, d3 = dj > 0 ? slotB : slotA;
            VTRACE(0);
            if (t > 0) {
                // ---- rows t-1 of the groups this row depends on
                wait_rows(t - 1u);
                VTRACE(1);
                // ---- lines entering from the neighbour CTAs: row t-1 of their edge column, into the ring slot of the entering lane
                if (enter1 | enter3) {
                    const unsigned pp = (t - 1u) & 1u, tag = ((t - 1u) >> 1) & 7u;
                    auto deposit = [&](const uint32_t *src, int path, int slot) {
                        // this warp's own pairs (relative to the sender part's minimum) and that minimum: all loads are issued
                        // before the first tag is checked (one L2 round trip when the line is already there)
                        const uint32_t *qm = src + K2 + part;
                        const int ka = k0 + lane, kb = ka + 32;                     // KP <= 64
                        uint32_t mu = ld_relaxed_gpu(qm);
                        uint32_t v0 = ka < k1 ? ld_relaxed_gpu(src + ka) : 0u, v1 = kb < k1 ? ld_relaxed_gpu(src + kb) : 0u;
                        if ((mu >> 28) != tag) mu = halo_wait2(qm, tag, abort_flag); else mu &= 0x0FFFFFFFu;
                        if (ka < k1) {
                            if ((v0 >> 28) != tag) v0 = halo_wait2(src + ka, tag, abort_flag); else v0 &= 0x0FFFFFFFu;
                            st[(path * K2 + ka) * NS + slot] = v0 + mu * 0x10001u;
                        }
                        if (kb < k1) {
                            if ((v1 >> 28) != tag) v1 = halo_wait2(src + kb, tag, abort_flag); else v1 &= 0x0FFFFFFFu;
                            st[(path * K2 + kb) * NS + slot] = v1 + mu * 0x10001u;
                        }
                        if (lane == 0) mn[(path * VPARTS + part) * NS + slot] = mu;
                    };
                    if (enter1) deposit(in1 + pp * HL, 0, __shfl_sync(0xFFFFFFFFu, d1, lane_leave3));
                    if (enter3) deposit(in3 + pp * HL, 2, __shfl_sync(0xFFFFFFFFu, d3, lane_leave1));
                    group_barrier();
                }
            }
            if (BAND && s == 0 && cont) {
                // ---- row band that continues a sweep: the predecessors of this row come from the state another band's sweep
                // exported (columns x - dj, x, x + dj of the row before the band), straight into the ring slots this row reads
                const uint32_t *imp = a.state_in + (long)f * a.state_words;
                const uint32_t *impm = imp + (long)3 * G32 * K2;
                const int xs[3] = {x - dj, x, x + dj};
                const int sl[3] = {d1, d2, d3};
#pragma unroll
                for (int pth = 0; pth < 3; pth++) {
                    if (xs[pth] >= 0 && xs[pth] < W) {
                        const uint32_t *src = imp + ((long)pth * G32 + xs[pth]) * K2;
                        for (int k = k0; k < k1; k++) st[(pth * K2 + k) * NS + sl[pth]] = src[k];
                        mn[(pth * VPARTS + part) * NS + sl[pth]] = impm[((long)pth * G32 + xs[pth]) * VPARTS + part];
                    }
                }
                p2w = p2_f[(long)i * G32];
                group_barrier();
            }
            VTRACE(2);
            const long tb0 = (((long)i * G + g) * K2 + k0) * 32;
            const uint16_t *cp = cost_f + tb0;
            SW *sp = S_f + tb0;
            if (s + 1 < H) {
                // pull the next row's operands of this warp into L2 while this row is being processed
                const long tbn = (((long)(i + di) * G + g) * K2 + k0) * 32 - lane;
                if (k0 + lane < k1) prefetch_l2(S_f + tbn + lane * 32);       // (RED: the line is in L2 when the reduction arrives)
                if (k0 + 2 * lane < k1) prefetch_l2(cost_f + tbn + lane * 64);
            }
            uint32_t *w1 = st + (0 * K2 + k0) * NS + d1, *w2 = st + (1 * K2 + k0) * NS + d2, *w3 = st + (2 * K2 + k0) * NS + d3;
            VPath2 p1, p2, p3;
            p1.mr = p2.mr = p3.mr = SW_INF2;
            if (s == 0 && !cont) {
                // first row of the pass: L = C on all three paths, nothing is summed (StereoSGM_SSE.hpp:116-218)
                for (int kb = k0; kb < k1; kb += VU) {
                    uint32_t cn[VU], sn[VU];
#pragma unroll
                    for (int u = 0; u < VU; u++) { cn[u] = 0; sn[u] = 0; }
                    if (kb + VU < k1) load_block(cp + VU * 32, nullptr, k1 - kb - VU, cn, sn, false);
#pragma unroll
                    for (int u = 0; u < VU; u++) {
                        if (FULL || kb + u < k1) {
                            const uint32_t c = __byte_perm(cb[u], 0, 0x4140);
                            w1[u * NS] = c; w2[u * NS] = c; w3[u * NS] = c;
                            p1.mr = __vminu2(p1.mr, c);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < VU; u++) cb[u] = cn[u];
                    cp += VU * 32; sp += VU * 32; w1 += VU * NS; w2 += VU * NS; w3 += VU * NS;
                }
                p2.mr = p1.mr; p3.mr = p1.mr;
            } else {
                // predecessors: r1 (i - di, x - dj), r2 (i - di, x), r3 (i - di, x + dj).  A line that enters through the image
                // border reads the border slot: L = 65535, min = 0 => L = C + P2 (StereoSGM_SSE.hpp:48-58,:69-72)
                const int r1s = border1 ? BIGS : d1, r3s = border3 ? BIGS : d3;
                const uint32_t *s1 = st + (0 * K2 + k0) * NS + r1s, *s2 = w2, *s3 = st + (2 * K2 + k0) * NS + r3s;
                uint32_t m1 = mn[(0 * VPARTS + 0) * NS + r1s], m2 = mn[(1 * VPARTS + 0) * NS + d2], m3 = mn[(2 * VPARTS + 0) * NS + r3s];
#pragma unroll
                for (int pt = 1; pt < VPARTS; pt++) {
                    m1 = min(m1, mn[(0 * VPARTS + pt) * NS + r1s]);
                    m2 = min(m2, mn[(1 * VPARTS + pt) * NS + d2]);
                    m3 = min(m3, mn[(2 * VPARTS + pt) * NS + r3s]);
                }
                p1.q = (m1 + (p2w & 0xFFu)) * 0x10001u;
                p2.q = (m2 + ((p2w >> 8) & 0xFFu)) * 0x10001u;
                p3.q = (m3 + (p2w >> 16)) * 0x10001u;
                p1.ng = m1; p2.ng = m2; p3.ng = m3;
                const uint32_t negm = 0u - ((m1 + m2) + m3) * 0x10001u;
                // the words just outside this warp's share are read before the other warps of the column group may overwrite them;
                // at the two ends of the disparity range they are the seams of the split-half packing:
                // below word 0: (inf, Lt[K2-1]) from word K2-1; above word K2-1: (Lt[K2], inf) from word 0
                const int ke = (k1 - k0) * NS, kt = (K2 - 1 - k0) * NS, kz = -k0 * NS;
                p1.prev = k0 > 0 ? s1[-NS] : __byte_perm(SW_INF2, s1[kt], 0x5410);
                p2.prev = k0 > 0 ? s2[-NS] : __byte_perm(SW_INF2, s2[kt], 0x5410);
                p3.prev = k0 > 0 ? s3[-NS] : __byte_perm(SW_INF2, s3[kt], 0x5410);
                const uint32_t wr1 = k1 < K2 ? s1[ke] : __byte_perm(s1[kz], SW_INF2, 0x5432),
                               wr2 = k1 < K2 ? s2[ke] : __byte_perm(s2[kz], SW_INF2, 0x5432),
                               wr3 = k1 < K2 ? s3[ke] : __byte_perm(s3[kz], SW_INF2, 0x5432);
                p1.cur = s1[0]; p2.cur = s2[0]; p3.cur = s3[0];
                group_barrier();                    // every warp of the group has read its neighbours' boundary pairs and minima
                VTRACE(3);
                int trb = 4;
                for (int kb = k0; kb < k1; kb += 2 * VU) {
                    uint32_t cn[VU], sn[VU];
                    const bool last1 = kb + VU >= k1;
                    if (!last1) load_block(cp + VU * 32, sp + VU * 32, k1 - kb - VU, cn, sn, true);
                    v2_block<NS, !FULL, NORM, RED>(cb, sb, s1, s2, s3, w1, w2, w3, wr1, wr2, wr3, p1, p2, p3, negm, p1x2, sp, k1 - kb, last1);
                    VTRACE(trb); trb++;
                    cp += VU * 32; sp += VU * 32;
                    s1 += VU * NS; s2 += VU * NS; s3 += VU * NS; w1 += VU * NS; w2 += VU * NS; w3 += VU * NS;
                    if (last1) break;
                    const bool last2 = kb + 2 * VU >= k1;
                    if (!last2) load_block(cp + VU * 32, sp + VU * 32, k1 - kb - 2 * VU, cb, sb, true);
                    v2_block<NS, !FULL, NORM, RED>(cn, sn, s1, s2, s3, w1, w2, w3, wr1, wr2, wr3, p1, p2, p3, negm, p1x2, sp, k1 - kb - VU, last2);
                    VTRACE(trb); trb++;
                    cp += VU * 32; sp += VU * 32;
                    s1 += VU * NS; s2 += VU * NS; s3 += VU * NS; w1 += VU * NS; w2 += VU * NS; w3 += VU * NS;
                }
            }
            // minima of this third of the row
            const uint32_t mr1 = min(p1.mr & 0xFFFFu, p1.mr >> 16), mr2 = min(p2.mr & 0xFFFFu, p2.mr >> 16),
                           mr3 = min(p3.mr & 0xFFFFu, p3.mr >> 16);
            mn[(0 * VPARTS + part) * NS + d1] = mr1;
            mn[(1 * VPARTS + part) * NS + d2] = mr2;
            mn[(2 * VPARTS + part) * NS + d3] = mr3;
            if (BAND && s == H - 1 && a.state_out != nullptr) {
                // ---- last row of a band: this column's new state of the three paths for the band that continues the sweep
                uint32_t *ex = a.state_out + (long)f * a.state_words;
                uint32_t *exm = ex + (long)3 * G32 * K2;
                const int sl[3] = {d1, d2, d3};
                const uint32_t mrs[3] = {mr1, mr2, mr3};
                __syncwarp();
#pragma unroll
                for (int pth = 0; pth < 3; pth++) {
                    uint32_t *dst = ex + ((long)pth * G32 + x) * K2;
                    for (int k = k0; k < k1; k++) dst[k] = st[(pth * K2 + k) * NS + sl[pth]];
                    exm[((long)pth * G32 + x) * VPARTS + part] = mrs[pth];
                }
            }
            // push the lines that leave the strip to the neighbour's inbound buffer of this row's parity: state relative to
            // this part's minimum (<= max C + P2 per half: the tag bits stay free), then the minimum itself
            const unsigned par = t & 1u;
            const uint32_t otag = ((t >> 1) & 7u) << 28;
            if (has1 && gl == gl_leave1) {
                __syncwarp();
                const int sl = __shfl_sync(0xFFFFFFFFu, d1, lane_leave1);
                const uint32_t mv = __shfl_sync(0xFFFFFFFFu, mr1, lane_leave1);
                uint32_t *dst = push1 + par * HL;
                for (int k = k0 + lane; k < k1; k += 32) st_relaxed_gpu(dst + k, (st[(0 * K2 + k) * NS + sl] - mv * 0x10001u) | otag);
                if (lane == 0) st_relaxed_gpu(dst + K2 + part, mv | otag);
            }
            if (has3 && gl == gl_leave3) {
                __syncwarp();
                const int sl = __shfl_sync(0xFFFFFFFFu, d3, lane_leave3);
                const uint32_t mv = __shfl_sync(0xFFFFFFFFu, mr3, lane_leave3);
                uint32_t *dst = push3 + par * HL;
                for (int k = k0 + lane; k < k1; k += 32) st_relaxed_gpu(dst + k, (st[(2 * K2 + k) * NS + sl] - mv * 0x10001u) | otag);
                if (lane == 0) st_relaxed_gpu(dst + K2 + part, mv | otag);
            }
            VTRACE(8);
            row_done(t);
            VTRACE(9);
            // prefetch for the next row: its P2 word and first operand block
            if (s + 1 < H) {
                const int in = i + di;
                p2w = p2_f[(long)in * G32];
                const long tbn = (((long)in * G + g) * K2 + k0) * 32;
                load_block(cost_f + tbn, S_f + tbn, k1 - k0, cb, sb, true);
            } else if (f + nteams < a.n) {
                const uint16_t *cost_n = cost_all + (long)(f + nteams) * a.t.frame + lane;
                const SW *S_n = reinterpret_cast<SW *>(S_all) + (long)(f + nteams) * a.t.frame + lane;
                load_block(cost_n + (((long)i1 * G + g) * K2 + k0) * 32, S_n + (((long)i1 * G + g) * K2 + k0) * 32, k1 - k0, cb, sb, cont);
            }
            VTRACE(10);
            if (++sh == n) sh = 0;
        }
    }
}

#ifdef VPP_TRACE
extern "C" int vppb200_debug_vtrace(unsigned long long *host, int n)
{
    return cudaMemcpyFromSymbol(host, g_vtrace, sizeof(unsigned long long) * (size_t)n) == cudaSuccess ? 0 : -1;
}
#endif

static size_t v_smem_bytes(int GC, int K2) { return ((size_t)3 * K2 * (GC * 32 + 1) + (size_t)3 * VPARTS * (GC * 32 + 1) + 4 + 4 * GC) * 4; }

// tuning / test hook: upper bound on the strip width in columns (0 = chosen by the planner)
static int g_max_strip = 0;
void sweep_set_max_strip(int cols) { g_max_strip = cols < 0 ? 0 : cols; }
static int g_force_teams = 0;       // experiment hook: frames in flight instead of the occupancy estimate
void sweep_set_clusters(int c) { g_force_teams = c < 0 ? 0 : c; }

// a team = the csize CTAs (one per SM) that hold one frame; nteams frames are in flight
struct VPlan { int csize, GC, nteams; size_t smem; };

template <int GC>
static int v_resident_ctas(size_t smem, int threads, int *out)
{
    int dev = 0, sms = 0, per_sm = 0;
    VPP_CUDA_TRY(cudaGetDevice(&dev));
    VPP_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    constexpr int NS = GC * 32 + 1;
    VPP_CUDA_TRY(cudaFuncSetAttribute(sgm_v2_kernel<NS, true, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VPP_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sgm_v2_kernel<NS, true, false, false, true>, threads, smem));
    // One CTA per SM.  (Measured: two CTAs of different frames per SM on 64-column strips take 3.83 us per row for their 4
    // column groups, one CTA with 5 groups 3.97 us -- the row time is a latency chain, wait -> hand-off -> setup -> loop ->
    // push, that does not shrink with the strip, so the widest strip that fits wins.)
    *out = per_sm >= 1 ? sms : 0;
    return VPPB200_OK;
}
static int v_resident(int GC, size_t smem, int *out)
{
    const int threads = GC * VPARTS * 32;
    switch (GC) {
        case 1: return v_resident_ctas<1>(smem, threads, out);
        case 2: return v_resident_ctas<2>(smem, threads, out);
        case 3: return v_resident_ctas<3>(smem, threads, out);
        case 4: return v_resident_ctas<4>(smem, threads, out);
        case 5: return v_resident_ctas<5>(smem, threads, out);
        default: return v_resident_ctas<5>(smem, threads, out);
    }
}

// Strip width: all CTAs of a team must be resident at once (they wait for each other's halo lines), so a team takes
// csize SMs and floor(#SM / csize) frames are in flight.  The planner minimises rounds x groups-per-CTA, i.e. the
// makespan of the launch in units of one 32-column group sweep.
// 0 = plan made; 1 = this shape does not fit the sweep; < 0 = error
static int plan_v(const TL &t, int n, VPlan *plan)
{
    // one-entry cache: the pipeline asks twice per call with the same shape
    static thread_local struct { int W, H, D, n, dev, strip, teams; VPlan p; bool ok; } memo = {0, 0, 0, 0, -1, 0, 0, {}, false};
    int dev = 0, smem_optin = 0, coop = 0;
    VPP_CUDA_TRY(cudaGetDevice(&dev));
    if (memo.ok && memo.W == t.W && memo.H == t.H && memo.D == t.D && memo.n == n && memo.dev == dev && memo.strip == g_max_strip &&
        memo.teams == g_force_teams) {
        *plan = memo.p;
        return VPPB200_OK;
    }
    VPP_CUDA_TRY(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    VPP_CUDA_TRY(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    if (!coop) return 1;
    if ((t.K2 + VPARTS - 1) / VPARTS > 64) return 1;     // the halo deposit moves at most two pairs per lane
    int gc_max = 0;
    for (int gc = 5; gc >= 1; gc--)
        if (v_smem_bytes(gc, t.K2) <= (size_t)smem_optin) { gc_max = gc; break; }
    if (g_max_strip > 0) gc_max = std::min(gc_max, std::max(1, g_max_strip / 32));
    if (gc_max < 1) return 1;
    long best_cost = -1;
    VPlan best{};
    for (int gc = gc_max; gc >= 1; gc--) {
        VPlan p;
        p.GC = gc;
        p.csize = (t.G + gc - 1) / gc;
        p.smem = v_smem_bytes(gc, t.K2);
        int resident = 0;
        int rc = v_resident(gc, p.smem, &resident);
        if (rc) return rc;
        int teams = resident / p.csize;
        if (teams < 1) continue;
        if (g_force_teams > 0) teams = std::min(teams, g_force_teams);
        p.nteams = std::min(teams, n);
        const long rounds = (n + p.nteams - 1) / p.nteams;
        // time of one round ~ max(1.6, 0.41 * gc) ms at K (measured on B200, tools/exp_clusters.py): below 4 groups the
        // SM is latency bound (too few warps), above it the round time grows with the strip width
        const long cost = rounds * std::max(160, 41 * gc);
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = p; }
        if (g_max_strip > 0) break;                 // forced strip width: take it as is
    }
    if (best_cost < 0) return 1;
    *plan = best;
    memo = {t.W, t.H, t.D, n, dev, g_max_strip, g_force_teams, best, true};
    return VPPB200_OK;
}

// A batch whose last round would leave most teams idle is swept in two launches: the first rounds with the widest strips, the
// rest with narrower strips and more CTAs per frame -- the row time falls with the strip width (measured at K, us per row: 3.97 /
// 3.67 / 3.50 / 3.40 for 5 / 4 / 3 / 2 column groups per CTA), so e.g. 64 K frames run as 36 frames x 8 CTAs (two rounds of 18
// teams) + 28 frames x 10 CTAs (two rounds of 14 teams) instead of four rounds of 18 teams with the last one 10 / 18 full.
struct VSplit { int n1; VPlan p1; int n2; VPlan p2; };
static int g_v_split = 1;
void sweep_set_v_split(int on) { g_v_split = on != 0; }
static int plan_v_split(const TL &t, int n, VSplit *out)
{
    static thread_local struct { int W, H, D, n, dev, strip, teams, split; VSplit s; bool ok; } memo = {0, 0, 0, 0, -1, 0, 0, 0, {}, false};
    int dev = 0;
    VPP_CUDA_TRY(cudaGetDevice(&dev));
    if (memo.ok && memo.W == t.W && memo.H == t.H && memo.D == t.D && memo.n == n && memo.dev == dev && memo.strip == g_max_strip &&
        memo.teams == g_force_teams && memo.split == g_v_split) {
        *out = memo.s;
        return VPPB200_OK;
    }
    VSplit best{};
    int rc = plan_v(t, n, &best.p1);
    if (rc) return rc;
    best.n1 = n; best.n2 = 0;
    if (g_v_split && g_max_strip == 0 && g_force_teams == 0 && n > best.p1.nteams) {
        static const double trow[6] = {0.0, 3.30, 3.40, 3.50, 3.67, 3.97};      // relative row time by groups per CTA
        const int gc_max = best.p1.GC;
        VPlan cand[6];
        bool have[6] = {false, false, false, false, false, false};
        for (int gc = 1; gc <= gc_max; gc++) {
            VPlan q;
            q.GC = gc; q.csize = (t.G + gc - 1) / gc; q.smem = v_smem_bytes(gc, t.K2);
            int resident = 0;
            if ((rc = v_resident(gc, q.smem, &resident))) return rc;
            q.nteams = resident / q.csize;
            if (q.nteams < 1) continue;
            cand[gc] = q; have[gc] = true;
        }
        auto rounds = [](int m, int teams) { return (m + teams - 1) / teams; };
        double best_cost = rounds(n, best.p1.nteams) * trow[best.p1.GC];
        const double launch = 0.05;                      // a second cooperative launch + P2 table, in the same units
        for (int a = 1; a <= gc_max; a++) {
            if (!have[a]) continue;
            for (int r1 = 1; r1 * cand[a].nteams < n; r1++) {
                const int n1 = r1 * cand[a].nteams, n2 = n - n1;
                for (int b = 1; b <= gc_max; b++) {
                    if (!have[b] || b == a) continue;
                    const double c = r1 * trow[a] + rounds(n2, cand[b].nteams) * trow[b] + launch;
                    if (c < best_cost - 1e-9) {
                        best_cost = c;
                        best.n1 = n1; best.p1 = cand[a]; best.p1.nteams = std::min(cand[a].nteams, n1);
                        best.n2 = n2; best.p2 = cand[b]; best.p2.nteams = std::min(cand[b].nteams, n2);
                    }
                }
            }
        }
    }
    *out = best;
    memo = {t.W, t.H, t.D, n, dev, g_max_strip, g_force_teams, g_v_split, best, true};
    return VPPB200_OK;
}

// the v-sweep's scratch behind the inbound halo lines: [abort flag (256 B)] [P2 table: n * H * G * 32 words]
static constexpr size_t HALO_LINES_BYTES = (size_t)1024 * 2 * 2 * (128 + 8) * 4;     // generously 1024 CTAs, D <= 256
size_t sweep_halo_bytes(int W, int H, int D, int n)
{
    (void)D;
    return HALO_LINES_BYTES + 256 + (size_t)n * H * ((W + 31) / 32) * 32 * 4;
}

static int g_v_red = 1;             // S += by red.global.add (default) instead of load + add + store
void sweep_set_v_red(int on) { g_v_red = on != 0; }

// words of one frame's exported row state: [3][G*32][K2] path words + [3][G*32][VPARTS] part minima
long sweep_state_words(int W, int D) { return (long)3 * ((W + 31) / 32) * 32 * (D / 2 + VPARTS); }

// a row band inside frames of Hfull rows (whole frame: row0 = 0, Hfull = t.H, pass_start = 1, no state hand-off)
struct VBand { int Hfull, row0, pass_start; const uint32_t *state_in; uint32_t *state_out; };

template <int GC>
static int run_v_t(const uint32_t *p2q, const uint16_t *cost, uint32_t *S, uint32_t *halo, uint32_t *abort_flag, const TL &t, int pass,
                   int n, const VPlan &p, bool norm, const VBand &band, const SgmParams &prm, cudaStream_t st)
{
    constexpr int NS = GC * 32 + 1;
    VArgs a;
    a.t = t; a.n = n; a.pass = pass; a.csize = p.csize; a.GC = p.GC;
    a.p1x2 = (uint32_t)prm.P1 * 0x10001u;
    a.pass_start = band.pass_start; a.state_in = band.state_in; a.state_out = band.state_out;
    a.state_words = sweep_state_words(t.W, t.D);
    // FULL: K2 splits into VPARTS equal shares of whole VU-blocks
    const bool full = t.K2 % (VPARTS * VU) == 0;
    void *args[] = {(void *)&p2q, (void *)&cost, (void *)&S, (void *)&halo, (void *)&abort_flag, (void *)&a};
    const bool banded = !band.pass_start || band.state_in != nullptr || band.state_out != nullptr;
    const void *kern;
#define VPP_VK(F, N, R) (banded ? (const void *)sgm_v2_kernel<NS, F, N, R, true> : (const void *)sgm_v2_kernel<NS, F, N, R, false>)
    if (norm && g_v_red) kern = full ? VPP_VK(true, true, true) : VPP_VK(false, true, true);
    else if (norm) kern = full ? VPP_VK(true, true, false) : VPP_VK(false, true, false);
    else if (g_v_red) kern = full ? VPP_VK(true, false, true) : VPP_VK(false, false, true);
    else kern = full ? VPP_VK(true, false, false) : VPP_VK(false, false, false);
#undef VPP_VK
    VPP_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    // cooperative launch: all CTAs resident (they poll each other's halo words), one grid sync at the start
    VPP_CUDA_TRY(cudaLaunchCooperativeKernel(kern, dim3((unsigned)(p.csize * p.nteams)), dim3((unsigned)(p.GC * VPARTS * 32)), args,
                                             p.smem, st));
    note_launch();
    return VPPB200_OK;
}

// norm: per-path normalisation (costs above the Hamming range, or frames too tall for the un-normalised state)
static int run_v(const uint8_t *img, const uint16_t *cost, uint32_t *S, void *halo_ws, const TL &t, int pass, int n,
                 const VPlan &p, bool norm, const SgmParams &prm, cudaStream_t st, const VBand *bandp = nullptr)
{
    const VBand band = bandp ? *bandp : VBand{t.H, 0, 1, nullptr, nullptr};
    uint32_t *halo = static_cast<uint32_t *>(halo_ws);
    uint32_t *abort_flag = nullptr;
    VPP_CUDA_TRY(cudaGetSymbolAddress(reinterpret_cast<void **>(&abort_flag), g_sweep_abort));
    uint32_t *p2q = reinterpret_cast<uint32_t *>(static_cast<char *>(halo_ws) + HALO_LINES_BYTES + 256);
    const int G32 = t.G * 32;
    // grid.y = frame * rows (<= 65535 per launch: whole frames per launch)
    if (t.H > 65535) return VPPB200_ERR_ARG;
    const int fpl = 65535 / t.H;
    for (int f0 = 0; f0 < n; f0 += fpl) {
        const int nf = std::min(fpl, n - f0);
        sgm_p2_kernel<<<dim3((unsigned)cdiv(G32 / 4, 256), (unsigned)(nf * t.H)), 256, 0, st>>>(
            img + (long)f0 * t.W * band.Hfull, p2q + (long)f0 * t.H * G32, t.W, band.Hfull, G32, pass, band.row0, t.H, prm);
        VPP_LAUNCH_CHECK("sgm_p2_kernel");
    }
    switch (p.GC) {
        case 1: return run_v_t<1>(p2q, cost, S, halo, abort_flag, t, pass, n, p, norm, band, prm, st);
        case 2: return run_v_t<2>(p2q, cost, S, halo, abort_flag, t, pass, n, p, norm, band, prm, st);
        case 3: return run_v_t<3>(p2q, cost, S, halo, abort_flag, t, pass, n, p, norm, band, prm, st);
        case 4: return run_v_t<4>(p2q, cost, S, halo, abort_flag, t, pass, n, p, norm, band, prm, st);
        default: return run_v_t<5>(p2q, cost, S, halo, abort_flag, t, pass, n, p, norm, band, prm, st);
    }
}

// 0 = no hand-off wait has timed out since the last call on the current device; 1 = one has (flag cleared).  Blocking.
int sweep_take_abort_flag(int *out)
{
    unsigned int v = 0, zero = 0;
    VPP_CUDA_TRY(cudaMemcpyFromSymbol(&v, g_sweep_abort, sizeof v));
    if (v) VPP_CUDA_TRY(cudaMemcpyToSymbol(g_sweep_abort, &zero, sizeof zero));
    *out = v != 0;
    return VPPB200_OK;
}

// does the sweep cover this shape on the current device?  (a team of resident CTAs must hold a frame's path state)
static int g_sweep_off = 0;
void sweep_set_enabled(int on) { g_sweep_off = !on; }
bool aggregate_tile_supported(int W, int H, int D, int n)
{
    if (g_sweep_off || H < 3) return false;
    const TL t = make_tl(W, H, D);
    if (t.frame >= (1L << 31)) return false;
    VPlan plan;
    return plan_v(t, n, &plan) == VPPB200_OK;
}

// The parameter domain of the sweeps (file header): with these the packed u16 arithmetic of the sweeps and of the fast per-path
// kernels never saturates, the P2 table's bytes hold P2 - P1, and the hand-off words keep their tag bits.  Outside it,
// compute_rsgm aggregates with the saturating generic kernels of sgm.cu.  Expects 0 <= P1, P2min, gamma <= 65535, alpha >= 0.
bool sweep_params_supported(const SgmParams &p, bool plain_costs)
{
    const int cmax = plain_costs ? 24 : 240;
    const int p2max = std::max(p.P2min, p.gamma);
    return p.P1 <= p.P2min && p2max - p.P1 <= 255 && cmax + p2max <= 4095;
}

// un-normalised v-sweep state (Hamming costs only): the running Lt <= 24 * H + P2max must stay inside uint16 (with slack; the
// default parameters give the 24 * H + 128 bound)
static bool v_norm(bool plain_costs, int H, const SgmParams &p)
{
    return !plain_costs || 24L * H + std::max(p.P2min, p.gamma) + 78 > 65535;
}

// 0 = done; 1 = this shape does not fit the sweep (caller uses sgm.cu); < 0 = error.
// dl != NULL: the last sweep is fused with the winner-takes-all step (left + sub-pixel into dl, right into dr) and the
// final S is never written; dl == NULL: S holds the aggregated volume in layout T.
// plain_costs: the costs are plain Hamming distances (<= 24, no guided modulation): the v-sweeps keep their path state
// un-normalised (see sgm_v2_kernel).
// (Two variants of round 1 were measured again on this kernel generation and removed: uint8 partial-sum volumes instead of one
// uint16 S -- 37 % less traffic, but the extra unpacking in the ALU-bound h-sweeps costs more than the v-sweeps gain, 25.4 vs
// 25.1 ms per step -- and a forward h-sweep that produces the cost volume itself, 5.27 ms vs 3.56 + 1.47 ms.)
// (Measured at the end of round 2 and removed: the forward h-sweep leaving its L as BYTE pairs -- <= 74 with Hamming costs -- and the
// first v-sweep writing S = that + its paths with plain stores: 11.8 GB less traffic per step, but the h-sweep's 16-byte pieces
// only bring it from 3.59 to 3.06 ms and the v-sweep with an operand load instead of the fire-and-forget reduction goes from 5.93 to
// 6.78 ms: step 22.3 vs 22.0 ms.)
int launch_aggregate_tile(const uint8_t *img, const uint8_t *cost8, uint16_t *S16, void *halo_ws, int W, int H, int D, int n,
                          float *dl, float *dr, const float *lut, bool plain_costs, const SgmParams &prm, const StageHook *hook,
                          cudaStream_t st)
{
    if (!sweep_params_supported(prm, plain_costs)) return VPPB200_ERR_ARG;
    const TL t = make_tl(W, H, D);
    VSplit sp;
    int rc = plan_v_split(t, n, &sp);
    if (rc) return rc;
    const uint16_t *cost = reinterpret_cast<const uint16_t *>(cost8);
    uint32_t *S = reinterpret_cast<uint32_t *>(S16);
    const bool norm = v_norm(plain_costs, H, prm);
    auto done = [&](int stage) { if (hook) hook->fn(hook->ctx, stage); };
    auto sweep = [&](int pass) -> int {
        int r = run_v(img, cost, S, halo_ws, t, pass, sp.n1, sp.p1, norm, prm, st);
        if (r == VPPB200_OK && sp.n2 > 0)
            r = run_v(img + (long)sp.n1 * t.W * t.H, cost + (long)sp.n1 * t.frame, S + (long)sp.n1 * t.frame, halo_ws, t, pass, sp.n2,
                      sp.p2, norm, prm, st);
        return r;
    };
    if ((rc = run_h(img, cost, S, t, 0, n, nullptr, nullptr, nullptr, prm, st))) return rc;
    done(VPPB200_STAGE_SGM_H_FWD);
    if ((rc = sweep(0))) return rc;
    done(VPPB200_STAGE_SGM_V_DOWN);
    if ((rc = sweep(1))) return rc;
    done(VPPB200_STAGE_SGM_V_UP);
    if ((rc = run_h(img, cost, S, t, dl ? 2 : 1, n, dl, dr, lut, prm, st))) return rc;
    done(VPPB200_STAGE_SGM_H_BWD);
    return VPPB200_OK;
}

// One row band [row0, row0 + rows) of frames of Hfull rows, for a frame that is split over several GPUs (SURVEY.md 8e row 5: the
// exact banded pipeline, not the reference's approximate StripedStereoSGM, RSGM/StereoSGM.h:116-133).  `phases` selects the
// steps to queue: COST (Hamming volume of the band from the full census images) | H_FWD | V_DOWN | V_UP | H_BWD (fused with WTA).
// The vertical sweeps continue across bands through the exported row state: V_DOWN of a band that does not start at row 0 reads
// state_in (= state_out of the band above), V_UP of a band that does not end at the last row reads state_in (= state_out of the
// band below); state_out == NULL: nothing is exported.  cost8 / S16 / dl / dr hold the band's rows only.
int launch_aggregate_band(const uint8_t *guide_full, const uint32_t *cen_l_full, const uint32_t *cen_r_full, uint8_t *cost8, uint16_t *S16,
                          void *halo_ws, int W, int Hfull, int D, int row0, int rows, int n, int phases, const uint32_t *state_in,
                          uint32_t *state_out, float *dl, float *dr, const float *lut, bool plain_costs, const SgmParams &prm,
                          cudaStream_t st)
{
    const TL t = make_tl(W, rows, D);
    if (row0 < 0 || rows < 3 || row0 + rows > Hfull) return VPPB200_ERR_ARG;
    if (!sweep_params_supported(prm, plain_costs)) return VPPB200_ERR_ARG;
    VPlan plan;
    int rc = plan_v(t, n, &plan);
    if (rc) return rc < 0 ? rc : VPPB200_ERR_ARG;
    const uint16_t *cost = reinterpret_cast<const uint16_t *>(cost8);
    uint32_t *S = reinterpret_cast<uint32_t *>(S16);
    const uint8_t *guide_band = guide_full + (long)row0 * W;       // the h-sweeps read the band's own rows of the guide (per frame: + f * W * Hfull)
    const bool norm = v_norm(plain_costs, Hfull, prm);
    if (n != 1 && Hfull != rows) {
        // frames are Hfull * W apart in the guide but rows * W apart in an h-sweep's row numbering: one frame per call when banded
        return VPPB200_ERR_ARG;
    }
    if (phases & 1) if ((rc = launch_cost_tile_band(cen_l_full, cen_r_full, cost8, W, Hfull, D, row0, rows, n, st))) return rc;
    if (phases & 2) if ((rc = run_h(guide_band, cost, S, t, 0, n, nullptr, nullptr, nullptr, prm, st))) return rc;
    if (phases & 4) {
        const VBand b{Hfull, row0, row0 == 0 ? 1 : 0, row0 == 0 ? nullptr : state_in, state_out};
        if (!b.pass_start && !state_in) return VPPB200_ERR_ARG;
        if ((rc = run_v(guide_full, cost, S, halo_ws, t, 0, n, plan, norm, prm, st, &b))) return rc;
    }
    if (phases & 8) {
        const bool last = row0 + rows == Hfull;
        const VBand b{Hfull, row0, last ? 1 : 0, last ? nullptr : state_in, state_out};
        if (!b.pass_start && !state_in) return VPPB200_ERR_ARG;
        if ((rc = run_v(guide_full, cost, S, halo_ws, t, 1, n, plan, norm, prm, st, &b))) return rc;
    }
    if (phases & 16) if ((rc = run_h(guide_band, cost, S, t, dl ? 2 : 1, n, dl, dr, lut, prm, st))) return rc;
    return VPPB200_OK;
}

// uint8 elements of a layout-T cost volume (S has the same number of uint16 elements)
size_t tile_volume_elems(int W, int H, int D, int n) { return (size_t)n * (size_t)make_tl(W, H, D).frame * 2; }

}  // namespace vppb200
