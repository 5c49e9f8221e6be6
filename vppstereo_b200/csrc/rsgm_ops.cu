// rsgm_ops.cu -- sm_100a kernels for every rSGM stage except the SGM aggregation itself (sgm.cu):
// padding + gray, 5x5 census, Hamming cost volume, WTA left/right (+ fused sub-pixel), median, gap interpolation,
// left-right check, speckle filter (connected components), background fill.
// Reference semantics: SURVEY.md Appendix A; file:line citations are relative to the reference root,
// RSGM/ = thirdparty/stereo-vision/reconstruction/base/rSGM/.  Compiled with -fmad=false (no FMA contraction).
#include "common.cuh"

namespace vppb200 {

// ------------------------------------------------------------------------------------------------------------
// padding (cv2.copyMakeBorder BORDER_REFLECT, models/rsgm/rsgm.py:258-260) fused with RGB2GRAY (rsgm.py:11-12)
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect_idx(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p - 1 : 2 * len - 1 - p;
    return p;
}

// gray[n][Hp][Wp]; OpenCV 4.13 RGB2GRAY = (R*9798 + G*19235 + B*3735 + 16384) >> 15.
// One thread = 4 adjacent output pixels of one padded row (Wp % 16 == 0), one 4-byte store; grid.y = frame * Hp + row.
__global__ void __launch_bounds__(128) pad_gray_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ gray, RsgmDims d)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q * 4 >= d.Wp) return;
    const long frow = blockIdx.y;                                  // f * Hp + y
    const int y = (int)(frow % d.Hp);
    const long f = frow / d.Hp;
    const int sy = reflect_idx(y - d.pt, d.H);
    const uint8_t *row = src + ((f * d.H + sy) * (long)d.W) * d.C;
    uint32_t out = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int sx = reflect_idx(q * 4 + i - d.pl, d.W);
        const uint8_t *p = row + (long)sx * d.C;
        uint32_t v;
        if (d.C == 3) v = (p[0] * 9798u + p[1] * 19235u + p[2] * 3735u + 16384u) >> 15;
        else v = p[0];
        out |= (v & 255u) << (8 * i);
    }
    reinterpret_cast<uint32_t *>(gray + frow * d.Wp)[q] = out;
}

// guide[n][Hp*Wp] = the first Hp*Wp BYTES of the padded interleaved image (RSGM/pyrSGM.cpp:586-588 reads a colour
// buffer as if it were gray).  One thread = 4 adjacent bytes (Hp*Wp % 4 == 0); grid.y = frame.
__global__ void __launch_bounds__(128) pad_flatbytes_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ guide, RsgmDims d)
{
    const unsigned np = (unsigned)d.Wp * (unsigned)d.Hp;
    const unsigned b0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4u;   // byte index inside the padded interleaved buffer
    if (b0 >= np) return;
    const long f = blockIdx.y;
    const uint8_t *img = src + f * (long)d.H * d.W * d.C;
    uint32_t out = 0;
    unsigned px = b0 / (unsigned)d.C, ch = b0 - px * (unsigned)d.C;
    unsigned y = px / (unsigned)d.Wp, x = px - y * (unsigned)d.Wp;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int sy = reflect_idx((int)y - d.pt, d.H), sx = reflect_idx((int)x - d.pl, d.W);
        out |= (uint32_t)img[((long)sy * d.W + sx) * d.C + ch] << (8 * i);
        if (++ch == (unsigned)d.C) { ch = 0; if (++x == (unsigned)d.Wp) { x = 0; y++; } }
    }
    reinterpret_cast<uint32_t *>(guide + f * (long)np)[b0 >> 2] = out;
}

int launch_pad_gray(const uint8_t *src, uint8_t *gray, const RsgmDims &d, int n, cudaStream_t st)
{
    const long rows = (long)n * d.Hp;
    if (d.Hp > 65535) return VPPB200_ERR_ARG;
    // grid.y is limited to 65535 rows: whole frames per launch
    for (long r0 = 0; r0 < rows; r0 += 65535 / d.Hp * (long)d.Hp) {      // whole frames per launch
        const long fr = r0 / d.Hp, nf = std::min((long)(65535 / d.Hp), n - fr);
        pad_gray_kernel<<<dim3(cdiv(d.Wp / 4, 128), (unsigned)(nf * d.Hp)), 128, 0, st>>>(src + fr * (long)d.H * d.W * d.C,
                                                                                      gray + fr * (long)d.Hp * d.Wp, d);
        VPP_LAUNCH_CHECK("pad_gray_kernel");
    }
    return VPPB200_OK;
}
int launch_pad_flatbytes(const uint8_t *src, uint8_t *guide, const RsgmDims &d, int n, cudaStream_t st)
{
    const long np = (long)d.Hp * d.Wp;
    for (int f0 = 0; f0 < n; f0 += 65535) {
        const int nf = std::min(65535, n - f0);
        pad_flatbytes_kernel<<<dim3(cdiv(np / 4, 128), nf), 128, 0, st>>>(src + f0 * (long)d.H * d.W * d.C, guide + f0 * np, d);
        VPP_LAUNCH_CHECK("pad_flatbytes_kernel");
    }
    return VPPB200_OK;
}

// ------------------------------------------------------------------------------------------------------------
// census5x5  (RSGM/FastFilters.cpp:181-442).  The image is a flat byte stream: neighbours of the first/last two
// columns wrap into the adjacent rows.  One thread produces 4 adjacent codes from 5 x 8 staged bytes; the four centres are compared
// against each neighbour offset with ONE byte-wise SIMD compare (__vsetltu4: 5 integer instructions for 4 comparisons).
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t census_tail_order(const uint8_t (&win)[5][8], int o)
{
    // scalar tail (:424-441): value = sum bit_k * 2^(23-k)
    const uint32_t c = win[2][o + 2];
    uint32_t v = 0;
#pragma unroll
    for (int dy = 0; dy < 5; dy++)
#pragma unroll
        for (int dx = 0; dx < 5; dx++) {
            if (dy == 2 && dx == 2) continue;
            v = v * 2 + (uint32_t)(c > win[dy][o + dx]);
        }
    return v;
}

__global__ void __launch_bounds__(256) census5x5_kernel(const uint8_t *__restrict__ src, uint32_t *__restrict__ dst, int W,
                                                        int H, long quads_per_frame, long total_quads)
{
    long q = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= total_quads) return;
    int qx, row;
    long f;
    split_fyx(q, W / 4, H, qx, row, f);                // (W % 16 == 0: the 4 centres share a row)
    const int col = qx * 4;
    const long c0 = (long)row * W + col;               // flat index of the first of 4 centres
    const long n = (long)W * H;
    const uint8_t *img = src + f * n;
    const long lo = 2L * W + 2, hi = (long)W * (H - 2) - 17;
    uint4 out = make_uint4(0, 0, 0, 0);
    const bool any_body = (c0 + 3 >= lo) && (c0 <= hi);
    const bool tail_row = (row == H - 3) && (col >= W - 16);
    if (any_body || tail_row) {
        // flat neighbours c0 + (dy-2)*W + (dx-2), dx = 0..7 (may wrap across row ends; outside the frame: 0), fetched as the
        // three aligned words that cover them (c0, W and n are multiples of 4: a word is entirely inside or outside)
        uint32_t wlo[5], whi[5];                       // window bytes 0..3 and 4..7 of each row = flat c0-2 .. c0+5
#pragma unroll
        for (int dy = 0; dy < 5; dy++) {
            const long a0 = c0 + (long)(dy - 2) * W - 4;
            uint32_t wd[3];
#pragma unroll
            for (int i = 0; i < 3; i++) {
                const long a = a0 + 4 * i;
                wd[i] = (a >= 0 && a < n) ? *reinterpret_cast<const uint32_t *>(img + a) : 0u;
            }
            wlo[dy] = __byte_perm(wd[0], wd[1], 0x5432); whi[dy] = __byte_perm(wd[1], wd[2], 0x5432);
        }
        // body pixels: the four centres are compared byte-wise in one register (neighbour < centre per byte), the 24 result
        // bits per pixel are shifted into three byte-sliced accumulators (neighbours 0-7, 8-15, 16-23: first neighbour = MSB,
        // the order of FastFilters.cpp:273-281) and transposed into the four codes at the end
        const uint32_t cw = __byte_perm(wlo[2], whi[2], 0x5432);
        uint32_t acc[3] = {0u, 0u, 0u};
        {
            int k = 0;
#pragma unroll
            for (int dy = 0; dy < 5; dy++)
#pragma unroll
                for (int dx = 0; dx < 5; dx++) {
                    if (dy == 2 && dx == 2) continue;
                    const uint32_t nb = __byte_perm(wlo[dy], whi[dy], 0x3210u + 0x1111u * dx);
                    acc[k / 8] = acc[k / 8] * 2u + __vsetltu4(nb, cw);
                    k++;
                }
        }
        uint32_t r[4];
#pragma unroll
        for (int o = 0; o < 4; o++) {
            const long c = c0 + o;
            const int cc = col + o;
            if (c >= lo && c <= hi) {
                r[o] = ((acc[0] >> (8 * o)) & 255u) | (((acc[1] >> (8 * o)) & 255u) << 8) | (((acc[2] >> (8 * o)) & 255u) << 16);
            } else if (row == H - 3 && cc >= W - 14 && cc <= W - 3) {
                uint8_t win[5][8];                     // (rare: the reference's scalar tail has its own bit order)
#pragma unroll
                for (int dy = 0; dy < 5; dy++)
#pragma unroll
                    for (int i = 0; i < 8; i++) win[dy][i] = (uint8_t)((i < 4 ? wlo[dy] : whi[dy]) >> (8 * (i & 3)));
                r[o] = census_tail_order(win, o);
            } else {
                r[o] = 0;
            }
        }
        out = make_uint4(r[0], r[1], r[2], r[3]);
    }
    reinterpret_cast<uint4 *>(dst + f * n)[c0 / 4] = out;
}

// ------------------------------------------------------------------------------------------------------------
// pad + RGB2GRAY + census5x5 in one kernel (the compute_rsgm front: rsgm.py:258-262 then FastFilters.cpp:181-442): the gray image
// never goes to HBM.  One CTA = CB_ROWS rows of the padded frame.  The source rows the band needs (its rows +-3, mapped back through
// BORDER_REFLECT: always one contiguous range of the interleaved uint8 image) arrive in shared memory as ONE bulk asynchronous
// copy (TMA engine, cp.async.bulk + mbarrier complete_tx; 16-byte aligned window around the range); the CTA converts them into the
// band's gray rows in shared memory (rows outside the frame = 0, which is what the flat-stream census reads there) and runs the
// same 4-codes-per-thread census as census5x5_kernel out of it.  Band height: 8 rows (70 KB per CTA at K).  16-row bands re-read less
// (22 source rows per 16 instead of 14 per 8: the kernel alone 0.14 vs 0.17 ms per 64 frames), but their 110 KB CTAs only fit on SMs
// that the v-sweeps of the neighbouring batch have left, and the pipelined step loses 0.5 ms (22.2 vs 21.7 ms); with 8 rows the step
// is where the two-kernel front was (21.7 ms), the gray image's round trip through HBM is gone and so is one launch per image.
// ------------------------------------------------------------------------------------------------------------
static constexpr int CB_ROWS = 8, CB_HALO = 3, CB_NT = 256, CB_BAND = CB_ROWS + 2 * CB_HALO;

__device__ __forceinline__ uint32_t cb_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__global__ void __launch_bounds__(CB_NT) census_fused_kernel(const uint8_t *__restrict__ src, uint32_t *__restrict__ dst, RsgmDims d,
                                                            long src_bytes, int bands, int raw_cap)
{
    extern __shared__ __align__(16) uint8_t csm[];
    uint8_t *raw = csm;                                            // [raw_cap] window of the source image
    uint8_t *gray = csm + raw_cap;                                 // [CB_BAND][Wp]
    uint64_t *mbar = reinterpret_cast<uint64_t *>(gray + CB_BAND * d.Wp);
    const int tid = threadIdx.x;
    const int band = blockIdx.x % bands;
    const long f = blockIdx.x / bands;
    const int W = d.Wp, H = d.Hp;
    const int y0 = band * CB_ROWS, ylo = y0 - CB_HALO;
    // source rows of the band (every thread: a dozen reflections)
    int sy_lo = d.H, sy_hi = -1;
    for (int r = 0; r < CB_BAND; r++) {
        const int yp = ylo + r;
        if (yp < 0 || yp >= H) continue;
        const int sy = reflect_idx(yp - d.pt, d.H);
        sy_lo = min(sy_lo, sy); sy_hi = max(sy_hi, sy);
    }
    const long row_bytes = (long)d.W * d.C;
    const long g_lo = (f * d.H + sy_lo) * row_bytes, g_hi = (f * d.H + sy_hi + 1) * row_bytes;     // byte range inside src
    const long a_lo = g_lo & ~15L;
    const long a_hi = min((g_hi + 15) & ~15L, src_bytes & ~15L);   // the bulk copy never reads past the tensor
    const int skew = (int)(g_lo - a_lo);
    const uint32_t mb = cb_smem_u32(mbar);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mb) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        const uint32_t bytes = (uint32_t)(a_hi - a_lo);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
        for (uint32_t off = 0; off < bytes; off += 32768u) {
            const uint32_t part = min(32768u, bytes - off);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(cb_smem_u32(raw + off)), "l"(src + a_lo + off), "r"(part), "r"(mb) : "memory");
        }
    }
    // (at most 15 bytes at the very end of the tensor are not covered by an aligned 16-byte piece)
    if (a_hi < g_hi && tid < (int)(g_hi - a_hi)) raw[(a_hi - a_lo) + tid] = src[a_hi + tid];
    {
        uint32_t ok = 0;
        while (!ok)
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(ok) : "r"(mb) : "memory");
    }
    __syncthreads();
    // the band's gray rows (cv2.copyMakeBorder BORDER_REFLECT + RGB2GRAY as pad_gray_kernel): a warp per row, 4 pixels per lane and
    // step; only the quads that touch the left / right border go through the reflection
    const int qw = W / 4;
    const int warp = tid >> 5, lane = tid & 31;
    for (int r = warp; r < CB_BAND; r += CB_NT / 32) {
        const int yp = ylo + r;
        uint32_t *grow = reinterpret_cast<uint32_t *>(gray + r * W);
        if (yp < 0 || yp >= H) {
            for (int q = lane; q < qw; q += 32) grow[q] = 0u;
            continue;
        }
        const uint8_t *rowp = raw + skew + (long)(reflect_idx(yp - d.pt, d.H) - sy_lo) * row_bytes;
        for (int q = lane; q < qw; q += 32) {
            const int sx0 = q * 4 - d.pl;
            const bool inner = sx0 >= 0 && sx0 + 3 < d.W;
            uint32_t out = 0;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const uint8_t *px = rowp + (inner ? sx0 + i : reflect_idx(sx0 + i, d.W)) * d.C;
                uint32_t v;
                if (d.C == 3) v = (px[0] * 9798u + px[1] * 19235u + px[2] * 3735u + 16384u) >> 15;
                else v = px[0];
                out |= (v & 255u) << (8 * i);
            }
            grow[q] = out;
        }
    }
    __syncthreads();
    // census of rows y0 .. y0 + CB_ROWS - 1 out of the band: flat index a of the frame = gray[a - ylo * W]
    const long n = (long)W * H;
    const long lo = 2L * W + 2, hi = (long)W * (H - 2) - 17;
    const uint8_t *img = gray - (long)ylo * W;
    for (int rr = warp; rr < CB_ROWS; rr += CB_NT / 32)
    for (int qx = lane; qx < qw; qx += 32) {
        const int row = y0 + rr, col = qx * 4;
        if (row >= H) break;
        const long c0 = (long)row * W + col;
        uint4 out = make_uint4(0, 0, 0, 0);
        const bool any_body = (c0 + 3 >= lo) && (c0 <= hi);
        const bool tail_row = (row == H - 3) && (col >= W - 16);
        if (any_body || tail_row) {
            uint32_t wlo[5], whi[5];
#pragma unroll
            for (int dy = 0; dy < 5; dy++) {
                const uint32_t *a0 = reinterpret_cast<const uint32_t *>(img + c0 + (long)(dy - 2) * W - 4);   // inside the band (halo 3)
                const uint32_t w0 = a0[0], w1 = a0[1], w2 = a0[2];
                wlo[dy] = __byte_perm(w0, w1, 0x5432); whi[dy] = __byte_perm(w1, w2, 0x5432);
            }
            const uint32_t cw = __byte_perm(wlo[2], whi[2], 0x5432);
            uint32_t acc[3] = {0u, 0u, 0u};
            {
                int k = 0;
#pragma unroll
                for (int dy = 0; dy < 5; dy++)
#pragma unroll
                    for (int dx = 0; dx < 5; dx++) {
                        if (dy == 2 && dx == 2) continue;
                        const uint32_t nb = __byte_perm(wlo[dy], whi[dy], 0x3210u + 0x1111u * dx);
                        acc[k / 8] = acc[k / 8] * 2u + __vsetltu4(nb, cw);
                        k++;
                    }
            }
            uint32_t r4[4];
#pragma unroll
            for (int o = 0; o < 4; o++) {
                const long c = c0 + o;
                const int cc = col + o;
                if (c >= lo && c <= hi) {
                    r4[o] = ((acc[0] >> (8 * o)) & 255u) | (((acc[1] >> (8 * o)) & 255u) << 8) | (((acc[2] >> (8 * o)) & 255u) << 16);
                } else if (row == H - 3 && cc >= W - 14 && cc <= W - 3) {
                    uint8_t win[5][8];
#pragma unroll
                    for (int dy = 0; dy < 5; dy++)
#pragma unroll
                        for (int i = 0; i < 8; i++) win[dy][i] = (uint8_t)((i < 4 ? wlo[dy] : whi[dy]) >> (8 * (i & 3)));
                    r4[o] = census_tail_order(win, o);
                } else {
                    r4[o] = 0;
                }
            }
            out = make_uint4(r4[0], r4[1], r4[2], r4[3]);
        }
        reinterpret_cast<uint4 *>(dst + f * n)[c0 / 4] = out;
    }
}

// 0 = done; 1 = not applicable here (source not 16-byte aligned, band beyond shared memory): the caller runs pad_gray + census
int launch_census_fused(const uint8_t *src, uint32_t *dst, const RsgmDims &d, int n, cudaStream_t st)
{
    if ((reinterpret_cast<uintptr_t>(src) & 15u) != 0 || d.Wp % 16 != 0) return 1;
    const long row_bytes = (long)d.W * d.C;
    const int raw_cap = (int)((CB_BAND * row_bytes + 32 + 15) & ~15L);
    const size_t smem = (size_t)raw_cap + (size_t)CB_BAND * d.Wp + 16;
    int dev = 0, smem_optin = 0;
    VPP_CUDA_TRY(cudaGetDevice(&dev));
    VPP_CUDA_TRY(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (smem > (size_t)smem_optin) return 1;
    const int bands = cdiv(d.Hp, CB_ROWS);
    if ((long)bands * n > 0x7FFFFFFFL) return 1;
    VPP_CUDA_TRY(cudaFuncSetAttribute(census_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    census_fused_kernel<<<(unsigned)(bands * n), CB_NT, smem, st>>>(src, dst, d, (long)n * d.H * row_bytes, bands, raw_cap);
    VPP_LAUNCH_CHECK("census_fused_kernel");
    return VPPB200_OK;
}

int launch_census(const uint8_t *src, uint32_t *dst, int W, int H, int n, cudaStream_t st)
{
    long qpf = (long)W * H / 4, total = qpf * n;
    census5x5_kernel<<<cdiv(total, 256), 256, 0, st>>>(src, dst, W, H, qpf, total);
    VPP_LAUNCH_CHECK("census5x5_kernel");
    return VPPB200_OK;
}

// ------------------------------------------------------------------------------------------------------------
// Hamming cost volume (RSGM/StereoBMHelper.cpp:29-140): rows 0,1,H-2,H-1 and d > x hold 12, else popc(L ^ R[x-d]).
// One thread = one pixel x 8 disparities = one 16-byte (u16) or 8-byte (u8) store.
// ------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) cost_kernel(const uint32_t *__restrict__ cl, const uint32_t *__restrict__ cr,
                                                   T *__restrict__ dsi, int W, int H, int D, long total)
{
    long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int d8 = D / 8;
    const int g = (int)(t % d8);
    const long px = t / d8;                    // pixel index over all frames
    const int x = (int)(px % W), y = (int)((px / W) % H);
    uint32_t v[8];
    if (y < 2 || y >= H - 2) {
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = 12;
    } else {
        const uint32_t l = cl[px];
        const uint32_t *rrow = cr + (px - x);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int d = g * 8 + k;
            v[k] = d > x ? 12u : (uint32_t)__popc(l ^ rrow[x - d]);
        }
    }
    if (sizeof(T) == 2) {
        uint4 o = make_uint4(v[0] | (v[1] << 16), v[2] | (v[3] << 16), v[4] | (v[5] << 16), v[6] | (v[7] << 16));
        reinterpret_cast<uint4 *>(dsi)[t] = o;
    } else {
        uint2 o = make_uint2(v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24), v[4] | (v[5] << 8) | (v[6] << 16) | (v[7] << 24));
        reinterpret_cast<uint2 *>(dsi)[t] = o;
    }
}

int launch_cost_u16(const uint32_t *cl, const uint32_t *cr, uint16_t *dsi, int W, int H, int D, int n, cudaStream_t st)
{
    long total = (long)n * H * W * (D / 8);
    cost_kernel<uint16_t><<<cdiv(total, 256), 256, 0, st>>>(cl, cr, dsi, W, H, D, total);
    VPP_LAUNCH_CHECK("cost_kernel<u16>");
    return VPPB200_OK;
}
int launch_cost_u8(const uint32_t *cl, const uint32_t *cr, uint8_t *dsi, int W, int H, int D, int n, cudaStream_t st)
{
    long total = (long)n * H * W * (D / 8);
    cost_kernel<uint8_t><<<cdiv(total, 256), 256, 0, st>>>(cl, cr, dsi, W, H, D, total);
    VPP_LAUNCH_CHECK("cost_kernel<u8>");
    return VPPB200_OK;
}

// _guided_dsi (models/rsgm/rsgm.py:115-127) on the u8 volume: numba evaluates the weight 10*(1-exp(-(h-d)^2/2)) in float64
// and rounds it to float32 once (fused array expression with a float32 result); dsi = (u16)((double)dsi * (double)w).
// Costs are <= 24 so the result is <= 240 and still fits uint8.  hints/valid are un-padded [n][H][W]; the padding
// region has validhints = 0 (BORDER_CONSTANT, rsgm.py:266-267).
__global__ void guided_u8_kernel(uint8_t *__restrict__ dsi, const float *__restrict__ hints, const float *__restrict__ valid,
                                 RsgmDims d, long total)
{
    long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int dd = (int)(t % d.D);
    const long px = t / d.D;
    const int x = (int)(px % d.Wp) - d.pl, y = (int)((px / d.Wp) % d.Hp) - d.pt;
    const long f = px / ((long)d.Wp * d.Hp);
    if (x < 0 || x >= d.W || y < 0 || y >= d.H) return;
    const long s = (f * d.H + y) * d.W + x;
    if (!(valid[s] > 0)) return;
    const double tt = __dsub_rn((double)hints[s], (double)dd);
    const float w = (float)__dmul_rn(10.0, __dsub_rn(1.0, exp(__ddiv_rn(-__dmul_rn(tt, tt), 2.0))));
    dsi[t] = (uint8_t)(uint16_t)__dmul_rn((double)dsi[t], (double)w);
}
int launch_guided_u8(uint8_t *dsi, const float *hints, const float *valid, const RsgmDims &d, int n, cudaStream_t st)
{
    long total = (long)n * d.Hp * d.Wp * d.D;
    guided_u8_kernel<<<cdiv(total, 256), 256, 0, st>>>(dsi, hints, valid, d, total);
    VPP_LAUNCH_CHECK("guided_u8_kernel");
    return VPPB200_OK;
}

// ------------------------------------------------------------------------------------------------------------
// Winner-takes-all.  One warp sweeps one image row from x = W-1 down to 0 and reads each S[y][x][:] exactly once
// (coalesced, lane l holds disparities [2*NW*l, 2*NW*(l+1)) ).
//   left  (RSGM/StereoBMHelper.cpp:634-750): first arg-min over d <= min(D-1, x): min over packed (cost<<16 | d).
//   right (:893-1015): disp_r[x] = first arg-min_k S[y][x+k][k].  A bucket per in-flight target pixel rides the lanes:
//          at column x' slot d holds target x'-d; after absorbing S[x'][d] every bucket moves one slot down, slot 0
//          retires to disp_r[x'].  No atomics, no re-reads.
//   sub-pixel (method 0, :1072-1102) optionally fused into the left result.
//   UNIQ: the uniqueness ratio uf (common.cuh: uniq_accept; left: a second warp reduction over the rivals of the arg-min, right:
//          the buckets carry uniq_absorb's state); a rejected pixel is -10 in both views.
//   INFO: (with UNIQ, any uf) the left pixel's best cost and least rival cost also go to info_cost / info_rival [rows][W].
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int s_at(const uint16_t *Srow, int x, int d, int D) { return Srow[(long)x * D + d]; }

template <int NW, bool LEFT, bool RIGHT, bool SUBPIX, bool UNIQ, bool INFO = false>
__device__ __forceinline__ void wta_rows_body(const uint16_t *__restrict__ S, float *__restrict__ disp_l, float *__restrict__ disp_r,
                                              int W, int H, int D, const float *__restrict__ lut, long total_rows, uint32_t uf,
                                              uint16_t *__restrict__ info_cost = nullptr, uint16_t *__restrict__ info_rival = nullptr)
{
    static_assert(!INFO || (UNIQ && LEFT), "the match info is the left view's uniqueness candidates");
    const long row = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= total_rows) return;
    const int lane = threadIdx.x & 31;
    const int d0 = 2 * NW * lane;
    const uint16_t *Srow = S + row * (long)W * D;
    const bool lane_valid = d0 < D;            // D % 8 == 0 and 2*NW in {2,4,6,8}: a lane is all-valid or partly valid
    uint32_t bucket[2 * NW];
#pragma unroll
    for (int k = 0; k < 2 * NW; k++) bucket[k] = 0xFFFFFFFFu;
    uint32_t bfr[UNIQ ? 2 * NW : 1], blast[UNIQ ? 2 * NW : 1];       // UNIQ: far | rest << 16 and the most recent cost per bucket
    if (UNIQ) {
#pragma unroll
        for (int k = 0; k < 2 * NW; k++) { bfr[k] = 0xFFFFFFFFu; blast[k] = 0xFFFFu; }
    }
    const bool last_image_row = false;
    (void)last_image_row;
    for (int x = W - 1; x >= 0; x--) {
        uint32_t key[2 * NW];
#pragma unroll
        for (int k = 0; k < NW; k++) {
            const int d = d0 + 2 * k;
            uint32_t w = 0xFFFFFFFFu;
            if (lane_valid && d < D) w = *reinterpret_cast<const uint32_t *>(Srow + (long)x * D + d);
            key[2 * k] = (d < D) ? ((w << 16) | (uint32_t)d) : 0xFFFFFFFFu;
            key[2 * k + 1] = (d + 1 < D) ? ((w & 0xFFFF0000u) | (uint32_t)(d + 1)) : 0xFFFFFFFFu;
        }
        if (LEFT) {
            const int end = min(D - 1, x);
            uint32_t m = 0xFFFFFFFFu;
#pragma unroll
            for (int k = 0; k < 2 * NW; k++) m = min(m, (d0 + k <= end) ? key[k] : 0xFFFFFFFFu);
            m = __reduce_min_sync(0xFFFFFFFFu, m);
            uint32_t c2 = 0xFFFFu;
            if (UNIQ) {
                const int b = (int)(m & 0xFFFFu);
#pragma unroll
                for (int k = 0; k < 2 * NW; k++) c2 = min(c2, uniq_rival(d0 + k, b, end) ? key[k] >> 16 : 0xFFFFu);
                c2 = __reduce_min_sync(0xFFFFFFFFu, c2);
            }
            if (lane == 0) {
                const int best = (int)(m & 0xFFFFu);
                float out = (float)best;
                if (SUBPIX && x >= 1 && x <= W - 2) {
                    if (best > 0) {
                        // best = D-1 reads the next pixel's d = 0 (xyd stream order)
                        const int c0 = s_at(Srow, x, best - 1, D), c1 = (int)(m >> 16);
                        const int c2 = best + 1 < D ? s_at(Srow, x, best + 1, D) : s_at(Srow, x + 1, 0, D);
                        const int lower = min(c1 - c0, c1 - c2);            // <= 0
                        out = __fadd_rn((float)best, __fmul_rn((float)(c2 - c0), lut[-lower]));
                    } else {
                        out = -10.0f;
                    }
                }
                if (UNIQ && !uniq_accept(m, c2, end, uf)) out = -10.0f;
                disp_l[row * W + x] = out;
                if (INFO) {
                    info_cost[row * W + x] = (uint16_t)(m >> 16);
                    info_rival[row * W + x] = (uint16_t)c2;
                }
            }
        }
        if (RIGHT) {
            if (UNIQ) {
#pragma unroll
                for (int k = 0; k < 2 * NW; k++) uniq_absorb(bucket[k], bfr[k], blast[k], key[k]);
            } else {
#pragma unroll
                for (int k = 0; k < 2 * NW; k++) bucket[k] = min(bucket[k], key[k]);
            }
            if (lane == 0) {
                float out = (float)(bucket[0] & 0xFFFFu);
                if (UNIQ && !uniq_accept(bucket[0], bfr[0] & 0xFFFFu, min(D - 1, W - 1 - x), uf)) out = -10.0f;
                disp_r[row * W + x] = out;
            }
            // shift every bucket one disparity slot down; the top slot of the warp starts a new target
            uint32_t from_up = __shfl_down_sync(0xFFFFFFFFu, bucket[0], 1);
            if (lane == 31) from_up = 0xFFFFFFFFu;
#pragma unroll
            for (int k = 0; k < 2 * NW - 1; k++) bucket[k] = bucket[k + 1];
            bucket[2 * NW - 1] = from_up;
            if (UNIQ) {
                uint32_t fr_up = __shfl_down_sync(0xFFFFFFFFu, bfr[0], 1), last_up = __shfl_down_sync(0xFFFFFFFFu, blast[0], 1);
                if (lane == 31) { fr_up = 0xFFFFFFFFu; last_up = 0xFFFFu; }
#pragma unroll
                for (int k = 0; k < 2 * NW - 1; k++) { bfr[k] = bfr[k + 1]; blast[k] = blast[k + 1]; }
                bfr[2 * NW - 1] = fr_up; blast[2 * NW - 1] = last_up;
            }
        }
    }
}

template <int NW, bool LEFT, bool RIGHT, bool SUBPIX>
__global__ void __launch_bounds__(128) wta_rows_kernel(const uint16_t *__restrict__ S, float *__restrict__ disp_l,
                                                       float *__restrict__ disp_r, int W, int H, int D,
                                                       const float *__restrict__ lut, long total_rows)
{
    wta_rows_body<NW, LEFT, RIGHT, SUBPIX, false>(S, disp_l, disp_r, W, H, D, lut, total_rows, UNIQ_OFF);
}
template <int NW, bool LEFT, bool RIGHT, bool SUBPIX>
__global__ void __launch_bounds__(128) wta_rows_uniq_kernel(const uint16_t *__restrict__ S, float *__restrict__ disp_l,
                                                            float *__restrict__ disp_r, int W, int H, int D,
                                                            const float *__restrict__ lut, long total_rows, uint32_t uf)
{
    wta_rows_body<NW, LEFT, RIGHT, SUBPIX, true>(S, disp_l, disp_r, W, H, D, lut, total_rows, uf);
}
// wta_rows_uniq_kernel (any uf, UNIQ_OFF included) exporting the left view's match info (compute_rsgm's volume paths)
template <int NW>
__global__ void __launch_bounds__(128) wta_rows_info_kernel(const uint16_t *__restrict__ S, float *__restrict__ disp_l,
                                                            float *__restrict__ disp_r, int W, int H, int D,
                                                            const float *__restrict__ lut, long total_rows, uint32_t uf,
                                                            uint16_t *__restrict__ info_cost, uint16_t *__restrict__ info_rival)
{
    wta_rows_body<NW, true, true, true, true, true>(S, disp_l, disp_r, W, H, D, lut, total_rows, uf, info_cost, info_rival);
}

template <bool LEFT, bool RIGHT, bool SUBPIX, bool UNIQ>
static int launch_wta_u(const uint16_t *S, float *dl, float *dr, int W, int H, int D, const float *lut, int n, uint32_t uf,
                        cudaStream_t st)
{
    const long rows = (long)n * H;
    const int blocks = cdiv(rows * 32, 128);
    const int nw = (D + 63) / 64;
#define VPP_WTA(NW)                                                                                                   \
    if (UNIQ) wta_rows_uniq_kernel<NW, LEFT, RIGHT, SUBPIX><<<blocks, 128, 0, st>>>(S, dl, dr, W, H, D, lut, rows, uf);     \
    else wta_rows_kernel<NW, LEFT, RIGHT, SUBPIX><<<blocks, 128, 0, st>>>(S, dl, dr, W, H, D, lut, rows);                 \
    break
    switch (nw) {
        case 1: VPP_WTA(1);
        case 2: VPP_WTA(2);
        case 3: VPP_WTA(3);
        default: VPP_WTA(4);
    }
#undef VPP_WTA
    VPP_LAUNCH_CHECK(UNIQ ? "wta_rows_uniq_kernel" : "wta_rows_kernel");
    return VPPB200_OK;
}
template <bool LEFT, bool RIGHT, bool SUBPIX>
static int launch_wta_t(const uint16_t *S, float *dl, float *dr, int W, int H, int D, const float *lut, int n, uint32_t uf,
                        cudaStream_t st)
{
    return uf < UNIQ_OFF ? launch_wta_u<LEFT, RIGHT, SUBPIX, true>(S, dl, dr, W, H, D, lut, n, uf, st)
                         : launch_wta_u<LEFT, RIGHT, SUBPIX, false>(S, dl, dr, W, H, D, lut, n, UNIQ_OFF, st);
}
int launch_wta_left(const uint16_t *S, float *disp, int W, int H, int D, int n, uint32_t uf, cudaStream_t st)
{
    return launch_wta_t<true, false, false>(S, disp, nullptr, W, H, D, nullptr, n, uf, st);
}
int launch_wta_right(const uint16_t *S, float *disp, int W, int H, int D, int n, uint32_t uf, cudaStream_t st)
{
    return launch_wta_t<false, true, false>(S, nullptr, disp, W, H, D, nullptr, n, uf, st);
}
int launch_wta_both_subpix(const uint16_t *S, float *dl, float *dr, int W, int H, int D, const float *lut, int n, uint32_t uf,
                           cudaStream_t st, uint16_t *info_cost, uint16_t *info_rival)
{
    if (!info_cost) return launch_wta_t<true, true, true>(S, dl, dr, W, H, D, lut, n, uf, st);
    const long rows = (long)n * H;
    const int blocks = cdiv(rows * 32, 128);
    switch ((D + 63) / 64) {
        case 1: wta_rows_info_kernel<1><<<blocks, 128, 0, st>>>(S, dl, dr, W, H, D, lut, rows, uf, info_cost, info_rival); break;
        case 2: wta_rows_info_kernel<2><<<blocks, 128, 0, st>>>(S, dl, dr, W, H, D, lut, rows, uf, info_cost, info_rival); break;
        case 3: wta_rows_info_kernel<3><<<blocks, 128, 0, st>>>(S, dl, dr, W, H, D, lut, rows, uf, info_cost, info_rival); break;
        default: wta_rows_info_kernel<4><<<blocks, 128, 0, st>>>(S, dl, dr, W, H, D, lut, rows, uf, info_cost, info_rival); break;
    }
    VPP_LAUNCH_CHECK("wta_rows_info_kernel");
    return VPPB200_OK;
}

// subPixelRefine as a stand-alone operator (RSGM/StereoBMHelper.cpp:1065-1135), one thread per pixel
__global__ void subpixel_kernel(const uint16_t *__restrict__ S, float *__restrict__ disp, int W, int H, int D, int method,
                                const float *__restrict__ lut, long total)
{
    long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int x = (int)(t % W);
    if (x < 1 || x > W - 2) return;
    const float v = disp[t];
    if (v > 0.0f) {
        const int dm = (int)v;
        const uint16_t *c = S + t * D + dm;
        const int c0 = c[-1], c1 = c[0], c2 = c[1];
        if (method == 0) {
            const int lower = min(c1 - c0, c1 - c2);
            // lower <= 0 whenever dm is the arg-min; for arbitrary input fall back to the table's 0 entry on positives
            const float r = lower <= 0 ? lut[-lower] : 0.0f;
            disp[t] = __fadd_rn((float)dm, __fmul_rn((float)(c2 - c0), r));
        } else {
            const int a = c0 + c0 - 4 * c1 + c2 + c2, b = c0 - c2;
            disp[t] = __fadd_rn((float)dm, __fdiv_rn((float)b, (float)a));
        }
    } else {
        disp[t] = -10.0f;
    }
}
int launch_subpixel(const uint16_t *S, float *disp, int W, int H, int D, int method, const float *lut, int n, cudaStream_t st)
{
    long total = (long)n * W * H;
    subpixel_kernel<<<cdiv(total, 256), 256, 0, st>>>(S, disp, W, H, D, method, lut, total);
    VPP_LAUNCH_CHECK("subpixel_kernel");
    return VPPB200_OK;
}

// ------------------------------------------------------------------------------------------------------------
// median3x3 (RSGM/FastFilters.cpp:701-757): flat-stream 3x3 median for c in [W+1, WH-W-5], copy elsewhere.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cswap(float &a, float &b) { float t = fminf(a, b); b = fmaxf(a, b); a = t; }

__device__ __forceinline__ float median9(float v0, float v1, float v2, float v3, float v4, float v5, float v6, float v7, float v8)
{
    cswap(v1, v2); cswap(v4, v5); cswap(v7, v8);
    cswap(v0, v1); cswap(v3, v4); cswap(v6, v7);
    cswap(v1, v2); cswap(v4, v5); cswap(v7, v8);
    cswap(v0, v3); cswap(v5, v8); cswap(v4, v7);
    cswap(v3, v6); cswap(v1, v4); cswap(v2, v5);
    cswap(v4, v7); cswap(v4, v2); cswap(v6, v4);
    cswap(v4, v2);
    return v4;
}

// one thread = 4 adjacent flat positions (W % 16 == 0, so W*H % 4 == 0): three 6-float windows, one float4 store; grid.y = frame
__global__ void __launch_bounds__(256) median3x3_kernel(const float *__restrict__ src, float *__restrict__ dst, int W, int H)
{
    const long n = (long)W * H;
    const long c0 = ((long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (c0 >= n) return;
    const float *s = src + (long)blockIdx.y * n;
    const float4 mid = *reinterpret_cast<const float4 *>(s + c0);
    float4 out = mid;
    if (c0 + 3 >= W + 1 && c0 <= n - W - 5) {
        // rows above / below exist for every position of the quad that is filtered (positions outside [W+1, n-W-5] keep
        // `mid`); the two flat neighbours beside the quad may lie outside the frame only for quads that are not filtered there
        const long up = c0 - W, dn = c0 + W;
        const bool has_up = up >= 0, has_dn = dn + 3 < n;
        float a[6], b[6], c[6];
        const float4 u4 = has_up ? *reinterpret_cast<const float4 *>(s + up) : make_float4(0, 0, 0, 0);
        const float4 d4 = has_dn ? *reinterpret_cast<const float4 *>(s + dn) : make_float4(0, 0, 0, 0);
        a[0] = (has_up && up >= 1) ? s[up - 1] : 0.0f; a[1] = u4.x; a[2] = u4.y; a[3] = u4.z; a[4] = u4.w; a[5] = has_up ? s[up + 4] : 0.0f;
        b[0] = c0 >= 1 ? s[c0 - 1] : 0.0f; b[1] = mid.x; b[2] = mid.y; b[3] = mid.z; b[4] = mid.w; b[5] = c0 + 4 < n ? s[c0 + 4] : 0.0f;
        c[0] = has_dn ? s[dn - 1] : 0.0f; c[1] = d4.x; c[2] = d4.y; c[3] = d4.z; c[4] = d4.w; c[5] = (has_dn && dn + 4 < n) ? s[dn + 4] : 0.0f;
        float r[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const long cc = c0 + i;
            r[i] = (cc < W + 1 || cc > n - W - 5) ? b[i + 1]
                                                  : median9(a[i], a[i + 1], a[i + 2], b[i], b[i + 1], b[i + 2], c[i], c[i + 1], c[i + 2]);
        }
        out = make_float4(r[0], r[1], r[2], r[3]);
    }
    *reinterpret_cast<float4 *>(dst + (long)blockIdx.y * n + c0) = out;
}
int launch_median(const float *src, float *dst, int W, int H, int n, cudaStream_t st)
{
    if (W % 4) return VPPB200_ERR_WIDTH;                       // (the operator requires W % 16 == 0 anyway)
    for (int f0 = 0; f0 < n; f0 += 65535) {
        const int nf = std::min(65535, n - f0);
        median3x3_kernel<<<dim3(cdiv((long)W * H / 4, 256), nf), 256, 0, st>>>(src + f0 * (long)W * H, dst + f0 * (long)W * H, W, H);
        VPP_LAUNCH_CHECK("median3x3_kernel");
    }
    return VPPB200_OK;
}

// ------------------------------------------------------------------------------------------------------------
// _linear_interpolate(dmap, 15, 3) + np.clip(., 0, None)   (models/rsgm/rsgm.py:66-113,:148-151)
// The reference scans a row left to right, in place: at a pixel <= 0 it looks for the nearest valid pixel within 7 on
// either side and, if both exist and differ by < 3, rewrites the whole span between them with the line through them.
// Closed form of that scan (exact): the span between two valid anchors is a maximal run of L invalid pixels; it is
// filled iff L <= 13 and |nl - nr| < 3, by the FIRST pixel of the run that sees both anchors, the one at position
// p = max(1, L - 6) (1-based): m = (nr - nl) / (L + 1), q = nl + m * p, value(j) = (float)(m * (j - p) + q) in float64.
// The rewritten anchors round back to themselves in float32, runs never chain (their anchors are original pixels), so
// every pixel is independent: one warp stages a row in shared memory, all lanes resolve their pixels, coalesced write.
// ------------------------------------------------------------------------------------------------------------
// INFO: the pixels of the crop [pt, pt+H) x [pl, pl+W) of state (cropped [n][H][W]) are set to VPPB200_STATE_INTERPOLATED where the
// map was <= 0 before this step (the value, if positive now, came from the interpolation), VPPB200_STATE_MATCHED elsewhere; the
// tail kernels overwrite the codes of the later stages.
template <bool INFO>
__device__ __forceinline__ void interp_clip_body(float *__restrict__ disp, int W, long total_rows, uint8_t *__restrict__ state,
                                                 const RsgmDims &d)
{
    extern __shared__ float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long row = (long)blockIdx.x * (blockDim.x >> 5) + warp;
    if (row >= total_rows) return;
    float *r = smem + (size_t)warp * W;
    float *g = disp + row * W;
    for (int x = lane; x < W; x += 32) r[x] = g[x];
    __syncwarp();
    for (int x = lane; x < W; x += 32) {
        float v = r[x];
        if (v <= 0) {
            int jl = 0, jr = 0;
            for (int k = 1; k <= 13 && x - k >= 0; k++)
                if (r[x - k] > 0) { jl = k; break; }
            if (jl)
                for (int k = 1; k <= 14 - jl && x + k < W; k++)
                    if (r[x + k] > 0) { jr = k; break; }
            if (jl && jr) {
                const int L = jl + jr - 1;                       // run length (<= 13), this pixel is number jl in it
                const double nl = r[x - jl], nr = r[x + jr];
                if (fabs(nl - nr) < 3.0) {
                    const int p = max(1, L - 6);
                    const double m = __ddiv_rn(nr - nl, (double)(L + 1));
                    const double q = __dsub_rn(nl, __dmul_rn(m, (double)(-p)));
                    v = (float)__dadd_rn(__dmul_rn(m, (double)(jl - p)), q);
                }
            }
        }
        g[x] = fmaxf(v, 0.0f);
        if (INFO) {
            const int y = (int)(row % d.Hp) - d.pt, xc = x - d.pl;
            if (y >= 0 && y < d.H && xc >= 0 && xc < d.W)
                state[((row / d.Hp) * d.H + y) * d.W + xc] = r[x] <= 0 ? VPPB200_STATE_INTERPOLATED : VPPB200_STATE_MATCHED;
        }
    }
}
__global__ void __launch_bounds__(128) interp_clip_kernel(float *__restrict__ disp, int W, long total_rows)
{
    interp_clip_body<false>(disp, W, total_rows, nullptr, RsgmDims{});
}
__global__ void __launch_bounds__(128) interp_clip_info_kernel(float *__restrict__ disp, long total_rows, uint8_t *__restrict__ state,
                                                               RsgmDims d)
{
    interp_clip_body<true>(disp, d.Wp, total_rows, state, d);
}
int launch_interp_clip(float *disp, int W, int H, int n, cudaStream_t st)
{
    const long rows = (long)n * H;
    const int wpb = 4;
    const size_t sm = (size_t)wpb * W * sizeof(float);
    if (sm > 48 * 1024) VPP_CUDA_TRY(cudaFuncSetAttribute(interp_clip_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    interp_clip_kernel<<<cdiv(rows, wpb), wpb * 32, sm, st>>>(disp, W, rows);
    VPP_LAUNCH_CHECK("interp_clip_kernel");
    return VPPB200_OK;
}
int launch_interp_clip_info(float *disp, const RsgmDims &d, int n, uint8_t *state, cudaStream_t st)
{
    const long rows = (long)n * d.Hp;
    const int wpb = 4;
    const size_t sm = (size_t)wpb * d.Wp * sizeof(float);
    if (sm > 48 * 1024) VPP_CUDA_TRY(cudaFuncSetAttribute(interp_clip_info_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    interp_clip_info_kernel<<<cdiv(rows, wpb), wpb * 32, sm, st>>>(disp, rows, state, d);
    VPP_LAUNCH_CHECK("interp_clip_info_kernel");
    return VPPB200_OK;
}

// ------------------------------------------------------------------------------------------------------------
// tail of compute_rsgm on the cropped H x W frame (models/rsgm/rsgm.py:275-292)
// ------------------------------------------------------------------------------------------------------------
// crop + _left_right_check(th=1) + zero mask==128 + astype(uint8)
// (u8, label and count rows have the stride Ws = W rounded up to 4, pad bytes 0, so that the speckle kernels can read words;
// the left-right check itself lives in speckle_rows_kernel)

// cv2.filterSpeckles(img, 0, 200, 10) (rsgm.py:285): 4-connected components under |a-b| <= 10 among non-zero pixels,
// components with <= 200 pixels are zeroed.  The relation is symmetric, so the labelling is order independent.
// Disparity maps are smooth: components are huge and rows consist of long runs.  Labelling therefore works on RUNS:
//   rows   : every pixel gets the index of the first pixel of its horizontal run (warp max-scan per row)
//   merge  : vertical links between runs by union-find (one union per pair of touching runs, not per pixel)
//   count  : one atomicAdd per run (its length) on the root
__device__ __forceinline__ bool spk_conn(int a, int b) { return a && b && abs(a - b) <= 10; }

// rows: crop + _left_right_check(th=1) + zero mask==128 + astype(uint8) (rsgm.py:229-248,:275-284) fused with the run labelling: the warp that labels a row
// produces the row's uint8 map itself (one pass over the two disparity rows instead of a kernel and a round trip of the map)
// INFO: state (cropped [n][H][W]) gets the code of the step that zeroes a pixel here: NO_MATCH (not positive), LR_REJECTED, BELOW_ONE
template <bool INFO>
__device__ __forceinline__ void speckle_rows_body(const float *__restrict__ dl, const float *__restrict__ dr, uint8_t *__restrict__ u8,
                                                  int *__restrict__ label, int *__restrict__ count, const RsgmDims &d, int Ws,
                                                  long total_rows, uint8_t *__restrict__ state)
{
    const long row = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= total_rows) return;
    const int lane = threadIdx.x & 31;
    const int W = d.W;
    const long base = row * Ws;
    const int y = (int)(row % d.H);
    const long f = row / d.H;
    const float *lrow = dl + ((f * d.Hp + y + d.pt) * d.Wp + d.pl);
    const float *rrow = dr + ((f * d.Hp + y + d.pt) * d.Wp + d.pl);
    int carry = 0;                                   // run start of the last pixel of the previous chunk
    int prev_last = 0;                               // uint8 value of the last pixel of the previous chunk
    for (int x0 = 0; x0 < Ws; x0 += 32) {
        const int x = x0 + lane;
        int v = 0;
        if (x < W) {
            float fv = lrow[x];
            int code = VPPB200_STATE_NO_MATCH;
            if (fv > 0) {
                code = VPPB200_STATE_BELOW_ONE;
                const int dd = __float2int_rn(fv);   // numba round(): half to even (rsgm.py:237)
                const int xd = x - dd;
                if (xd >= 0 && xd <= W - 1) {
                    const float r = rrow[xd];
                    if (r > 0 && fabsf(__fsub_rn(fv, r)) > 1.0f) { fv = 0.0f; code = VPPB200_STATE_LR_REJECTED; }
                } else {
                    fv = 0.0f;
                    code = VPPB200_STATE_LR_REJECTED;
                }
            }
            v = (int)(uint8_t)fv;
            if (INFO && !v) state[row * W + x] = (uint8_t)code;
        }
        int left = __shfl_up_sync(0xFFFFFFFFu, v, 1);
        if (lane == 0) left = prev_last;
        prev_last = __shfl_sync(0xFFFFFFFFu, v, 31);
        int s = spk_conn(v, left) ? -1 : x;          // -1: continues the run of the pixel to the left
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xFFFFFFFFu, s, o);
            if (lane >= o) s = max(s, t);
        }
        if (s < 0) s = carry;
        carry = __shfl_sync(0xFFFFFFFFu, s, 31);
        if (x < Ws) u8[base + x] = (uint8_t)v;       // (pad bytes of the row stride: 0)
        if (x < W) {
            label[base + x] = v ? (int)(base + s) : -1;
            count[base + x] = 0;
        }
    }
}
__global__ void __launch_bounds__(128) speckle_rows_kernel(const float *__restrict__ dl, const float *__restrict__ dr,
                                                           uint8_t *__restrict__ u8, int *__restrict__ label,
                                                           int *__restrict__ count, RsgmDims d, int Ws, long total_rows)
{
    speckle_rows_body<false>(dl, dr, u8, label, count, d, Ws, total_rows, nullptr);
}
__global__ void __launch_bounds__(128) speckle_rows_info_kernel(const float *__restrict__ dl, const float *__restrict__ dr,
                                                                uint8_t *__restrict__ u8, int *__restrict__ label,
                                                                int *__restrict__ count, RsgmDims d, int Ws, long total_rows,
                                                                uint8_t *__restrict__ state)
{
    speckle_rows_body<true>(dl, dr, u8, label, count, d, Ws, total_rows, state);
}

__device__ __forceinline__ int uf_find(const int *L, int i)
{
    int p = L[i];
    while (p != i) { i = p; p = L[i]; }
    return i;
}
__device__ __forceinline__ int uf_find_compress(int *L, int i)
{
    const int r = uf_find(L, i);
    while (i != r) { const int nx = L[i]; L[i] = r; i = nx; }   // only used when no union runs concurrently
    return r;
}
// find with path halving.  Parent pointers only ever decrease (the larger root is linked under the smaller one), so
// L[i] = grandparent always stores a valid ancestor; racing with a concurrent union it can at worst undo a link that
// union's own retry loop re-establishes (the scheme of ECL-CC).
__device__ __forceinline__ int uf_find_halve(int *L, int i)
{
    int p = L[i];
    while (p != i) {
        const int gp = L[p];
        if (gp != p) L[i] = gp;
        i = p; p = gp;
    }
    return i;
}
__device__ __forceinline__ void uf_union(int *L, int a, int b)
{
    bool done = false;
    while (!done) {
        a = uf_find_halve(L, a);
        b = uf_find_halve(L, b);
        if (a < b) { int old = atomicMin(&L[b], a); done = (old == b); b = old; }
        else if (b < a) { int old = atomicMin(&L[a], b); done = (old == a); a = old; }
        else done = true;
    }
}
// one thread = 4 adjacent pixels of a row: the row's word, the word below and the two bytes to their left
__global__ void __launch_bounds__(256) speckle_merge_kernel(const uint8_t *__restrict__ u8, int *label, int W, int Ws, int H, long total_quads)
{
    const long q = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= total_quads) return;
    const unsigned qpr = (unsigned)Ws >> 2;                    // (the launcher guarantees total_quads < 2^31)
    const long row = (long)((unsigned)q / qpr);
    const int x0 = (int)((unsigned)q - (unsigned)row * qpr) * 4;
    if ((int)(row % H) + 1 >= H) return;
    const long t0 = row * Ws + x0;
    const uint32_t w0 = *reinterpret_cast<const uint32_t *>(u8 + t0);
    if (!w0) return;
    const uint32_t w1 = *reinterpret_cast<const uint32_t *>(u8 + t0 + Ws);
    if (!w1) return;
    int vl = x0 > 0 ? u8[t0 - 1] : 0, ql = x0 > 0 ? u8[t0 + Ws - 1] : 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int v = (w0 >> (8 * i)) & 255, qv = (w1 >> (8 * i)) & 255;
        // (x > 0: the same pair of runs is already linked through the column to the left)
        if (spk_conn(v, qv) && !(x0 + i > 0 && spk_conn(vl, v) && spk_conn(ql, qv) && spk_conn(vl, ql)))
            uf_union(label, label[t0 + i], label[t0 + Ws + i]);
        vl = v; ql = qv;
    }
}
__global__ void __launch_bounds__(256) speckle_count_kernel(const uint8_t *__restrict__ u8, int *label, int *count, int W, int Ws, long total_quads)
{
    const long q = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= total_quads) return;
    const unsigned qpr = (unsigned)Ws >> 2;                    // (the launcher guarantees total_quads < 2^31)
    const long row = (long)((unsigned)q / qpr);
    const int x0 = (int)((unsigned)q - (unsigned)row * qpr) * 4;
    const long t0 = row * Ws + x0;
    const uint32_t w0 = *reinterpret_cast<const uint32_t *>(u8 + t0);
    if (!w0) return;
    int prev = x0 > 0 ? u8[t0 - 1] : 0;
    const int after = x0 + 4 < W ? u8[t0 + 4] : 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int x = x0 + i;
        const int v = (w0 >> (8 * i)) & 255;
        const int next = i < 3 ? (int)((w0 >> (8 * i + 8)) & 255) : after;
        if (v && x < W) {
            const bool run_end = (x == W - 1) || !spk_conn(v, next);
            if (run_end) {
                // first pixel of this run: a non-start pixel still holds it (row kernel); a start pixel's own label may
                // already point at another run's root, so a one-pixel run must not read its length from it
                const bool is_start = (x == 0) || !spk_conn(prev, v);
                const long t = t0 + i;
                const int start = is_start ? (int)t : label[t];
                const int root = uf_find_compress(label, start);
                atomicAdd(&count[root], (int)(t - start) + 1);
            }
        }
        prev = v;
    }
}
// apply the speckle verdict, restore sub-pixel values (rsgm.py:286-290) and write the float frame
// INFO: a speckle gets VPPB200_STATE_SPECKLE (every other code is already in state), and the padded cost / rival maps are cropped
// into cost_out / rival_out
template <bool INFO>
__device__ __forceinline__ void speckle_apply_body(const uint8_t *__restrict__ u8, const int *__restrict__ label,
                                                   const int *__restrict__ count, const float *__restrict__ dl, float *__restrict__ out,
                                                   const RsgmDims &d, int Ws, int subpixel, long total, uint8_t *__restrict__ state,
                                                   const uint16_t *__restrict__ cost_pad, const uint16_t *__restrict__ rival_pad,
                                                   uint16_t *__restrict__ cost_out, uint16_t *__restrict__ rival_out)
{
    long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    int x, y;
    long f;
    split_fyx(t, d.W, d.H, x, y, f);
    const long ts = (f * d.H + y) * Ws + x;
    int b = u8[ts];
    if (b) {
        const int start = label[ts];                  // a non-start pixel still holds its run start
        const int root = uf_find(label, start);
        if (count[root] <= 200) {
            b = 0;
            if (INFO) state[t] = VPPB200_STATE_SPECKLE;
        }
    }
    float v = (float)b;
    if (subpixel && b) v = dl[(f * d.Hp + y + d.pt) * d.Wp + d.pl + x];
    out[t] = v;
    if (INFO) {
        const long tp = (f * d.Hp + y + d.pt) * d.Wp + d.pl + x;
        cost_out[t] = cost_pad[tp];
        rival_out[t] = rival_pad[tp];
    }
}
__global__ void speckle_apply_kernel(const uint8_t *__restrict__ u8, const int *__restrict__ label, const int *__restrict__ count,
                                     const float *__restrict__ dl, float *__restrict__ out, RsgmDims d, int Ws, int subpixel,
                                     long total)
{
    speckle_apply_body<false>(u8, label, count, dl, out, d, Ws, subpixel, total, nullptr, nullptr, nullptr, nullptr, nullptr);
}
__global__ void speckle_apply_info_kernel(const uint8_t *__restrict__ u8, const int *__restrict__ label, const int *__restrict__ count,
                                          const float *__restrict__ dl, float *__restrict__ out, RsgmDims d, int Ws, int subpixel,
                                          long total, uint8_t *__restrict__ state, const uint16_t *__restrict__ cost_pad,
                                          const uint16_t *__restrict__ rival_pad, uint16_t *__restrict__ cost_out,
                                          uint16_t *__restrict__ rival_out)
{
    speckle_apply_body<true>(u8, label, count, dl, out, d, Ws, subpixel, total, state, cost_pad, rival_pad, cost_out, rival_out);
}

// _interpolate_background rows (rsgm.py:188-213).  Closed form of the sequential scan (exact): an invalid run with valid
// pixels on both sides takes the minimum of the two, a run that touches the left (right) border takes the first (last)
// valid value of the row, a row without valid pixels stays as it is; fills only ever read ORIGINAL valid pixels.  One
// warp per row staged in shared memory: nearest valid index to the left by a ballot scan over 32-pixel chunks, then the
// same from the right while writing the result.
__global__ void __launch_bounds__(128) bg_rows_kernel(float *__restrict__ img, int W, long total_rows)
{
    extern __shared__ float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long row = (long)blockIdx.x * (blockDim.x >> 5) + warp;
    if (row >= total_rows) return;
    float *r = smem + (size_t)warp * 2 * W;
    int *pv = reinterpret_cast<int *>(r + W);        // index of the nearest valid pixel to the left (-1: none)
    float *g = img + row * W;
    for (int x = lane; x < W; x += 32) r[x] = g[x];
    __syncwarp();
    int carry = -1;
    for (int x0 = 0; x0 < W; x0 += 32) {
        const int x = x0 + lane;
        const bool valid = x < W && r[x] > 0;
        const unsigned m = __ballot_sync(0xFFFFFFFFu, valid);
        const unsigned lower = m & ((1u << lane) - 1u);
        if (x < W) pv[x] = lower ? x0 + 31 - __clz(lower) : carry;
        if (m) carry = x0 + 31 - __clz(m);
    }
    __syncwarp();
    carry = W;                                       // nearest valid pixel to the right (W: none)
    for (int x0 = ((W - 1) / 32) * 32; x0 >= 0; x0 -= 32) {
        const int x = x0 + lane;
        const bool valid = x < W && r[x] > 0;
        const unsigned m = __ballot_sync(0xFFFFFFFFu, valid);
        if (x < W && !valid) {
            const unsigned upper = lane == 31 ? 0u : (m >> (lane + 1)) << (lane + 1);
            const int nv = upper ? x0 + __ffs(upper) - 1 : carry;
            const int lv = pv[x];
            float out = r[x];
            if (lv >= 0 && nv < W) out = fminf(r[lv], r[nv]);
            else if (lv >= 0) out = r[lv];
            else if (nv < W) out = r[nv];
            g[x] = out;
        }
        if (m) carry = x0 + __ffs(m) - 1;
    }
}
// _interpolate_background columns (rsgm.py:215-227): thread per column (coalesced across the warp)
__global__ void bg_cols_kernel(float *__restrict__ img, int W, int H, long total_cols)
{
    long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total_cols) return;
    const int u = (int)(t % W);
    float *col = img + (t / W) * (long)W * H + u;
    for (int v = 0; v < H; v++)
        if (col[(long)v * W] > 0) { const float f = col[(long)v * W]; for (int v2 = 0; v2 < v; v2++) col[(long)v2 * W] = f; break; }
    for (int v = H - 1; v >= 0; v--)
        if (col[(long)v * W] > 0) { const float f = col[(long)v * W]; for (int v2 = v + 1; v2 < H; v2++) col[(long)v2 * W] = f; break; }
}

// info: NULL (the default launches) or the match info's outputs (launch_tail_info)
struct TailInfo { uint8_t *state; const uint16_t *cost_pad, *rival_pad; uint16_t *cost_out, *rival_out; };
static int tail_impl(const float *dl, const float *dr, float *out, const RsgmDims &d, int subpixel, TailBufs tb, int n,
                     const TailInfo *info, cudaStream_t st)
{
    const long total = (long)n * d.H * d.W;
    if ((long)n * d.H * tail_stride(d.W) >= (1L << 31)) return VPPB200_ERR_ARG;
    const int blocks = cdiv(total, 256);
    const int Ws = tail_stride(d.W);
    const long quads = (long)n * d.H * (Ws >> 2);
    {
        const long nrows = (long)n * d.H;
        if (info) {
            speckle_rows_info_kernel<<<cdiv(nrows * 32, 128), 128, 0, st>>>(dl, dr, tb.u8, tb.label, tb.count, d, Ws, nrows, info->state);
            VPP_LAUNCH_CHECK("speckle_rows_info_kernel");
        } else {
            speckle_rows_kernel<<<cdiv(nrows * 32, 128), 128, 0, st>>>(dl, dr, tb.u8, tb.label, tb.count, d, Ws, nrows);
            VPP_LAUNCH_CHECK("speckle_rows_kernel");
        }
    }
    speckle_merge_kernel<<<cdiv(quads, 256), 256, 0, st>>>(tb.u8, tb.label, d.W, Ws, d.H, quads);
    VPP_LAUNCH_CHECK("speckle_merge_kernel");
    speckle_count_kernel<<<cdiv(quads, 256), 256, 0, st>>>(tb.u8, tb.label, tb.count, d.W, Ws, quads);
    VPP_LAUNCH_CHECK("speckle_count_kernel");
    if (info) {
        speckle_apply_info_kernel<<<blocks, 256, 0, st>>>(tb.u8, tb.label, tb.count, dl, out, d, Ws, subpixel, total, info->state,
                                                          info->cost_pad, info->rival_pad, info->cost_out, info->rival_out);
        VPP_LAUNCH_CHECK("speckle_apply_info_kernel");
    } else {
        speckle_apply_kernel<<<blocks, 256, 0, st>>>(tb.u8, tb.label, tb.count, dl, out, d, Ws, subpixel, total);
        VPP_LAUNCH_CHECK("speckle_apply_kernel");
    }
    const long rows = (long)n * d.H;
    const int wpb = 4;
    const size_t sm = (size_t)wpb * 2 * d.W * sizeof(float);
    if (sm > 48 * 1024) VPP_CUDA_TRY(cudaFuncSetAttribute(bg_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    bg_rows_kernel<<<cdiv(rows, wpb), wpb * 32, sm, st>>>(out, d.W, rows);
    VPP_LAUNCH_CHECK("bg_rows_kernel");
    const long cols = (long)n * d.W;
    bg_cols_kernel<<<cdiv(cols, 128), 128, 0, st>>>(out, d.W, d.H, cols);
    VPP_LAUNCH_CHECK("bg_cols_kernel");
    return VPPB200_OK;
}
int launch_tail(const float *dl, const float *dr, float *out, const RsgmDims &d, int subpixel, TailBufs tb, int n, cudaStream_t st)
{
    return tail_impl(dl, dr, out, d, subpixel, tb, n, nullptr, st);
}
int launch_tail_info(const float *dl, const float *dr, float *out, const RsgmDims &d, int subpixel, TailBufs tb, int n, uint8_t *state,
                     const uint16_t *cost_pad, const uint16_t *rival_pad, uint16_t *cost_out, uint16_t *rival_out, cudaStream_t st)
{
    const TailInfo info{state, cost_pad, rival_pad, cost_out, rival_out};
    return tail_impl(dl, dr, out, d, subpixel, tb, n, &info, st);
}

}  // namespace vppb200
