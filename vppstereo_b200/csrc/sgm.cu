// sgm.cu -- 8-path SGM aggregation on sm_100a, bit-exact with the reference's raster recursion
// (RSGM/StereoSGM_SSE.hpp:13-515 via RSGM/pyrSGM.cpp:504-637; semantics in SURVEY.md A.4).
//
// Decomposition.  The reference sweeps the image twice (pass 0 top-down/left-right, pass 1 mirrored) and updates
// four paths per pixel inside each sweep.  Every path is a family of independent 1-D recurrences, so here one WARP
// owns one path line and walks it; lane l holds disparities [2*NW*l, 2*NW*(l+1)) packed two per register (u16x2).
//   r0 (horizontal) : one line per row, L(j1) = C
//   r2 (vertical)   : one line per column, starts on the pass's first row with L = C (not summed into S, :116-218)
//   r1, r3 (diagonal): lines that start on the first row behave like r2; lines that enter through a side column
//                     start from the border slot L = 65535, min = 0, i.e. L = C + P2 (:48-58,:69-72)
// Reproduced quirks: P2 intensities are read from the FLAT image stream (wrap across row ends); on the row right
// after a pass's first row the "previous line" is that same row (:221); row H-1 of pass 1 adds with uint16
// wrap-around (:143,:198); everything else saturates at 65535.
//
// Two instantiations:
//   fast    : uint8 costs, parameters inside the sweep domain (sweep_params_supported in sgm_sweep.cu: L <= Cmax + P2max,
//             S <= 8 * (Cmax + P2max) < 65536), DPX-style packed min/add (VIMNMX/VIADDMNMX.U16x2); no saturation is
//             reachable; used by compute_rsgm for shapes the sweeps cannot hold;
//   generic : uint16 costs (the aggregate_SSE drop-in) or the uint8 volume of compute_rsgm (parameters outside the sweep
//             domain), arbitrary parameters, explicit saturation.
#include "common.cuh"

namespace vppb200 {

struct SgmArgs {
    int W, H, D;
    SgmParams p;
    int r;          // path 0..3
    int pass;       // 0 / 1
    int lines;      // lines per frame
};

struct LineGeom {
    int i, j;        // start pixel
    int si, sj;      // step
    int len;         // pixels on the line
    bool border;     // true: predecessor of the start pixel is the out-of-image border slot
    int i1, di, dj;
};

__device__ __forceinline__ LineGeom line_geom(const SgmArgs &a, int id)
{
    LineGeom g;
    g.di = a.pass == 0 ? 1 : -1;
    g.dj = g.di;
    g.i1 = a.pass == 0 ? 0 : a.H - 1;
    const int j1 = a.pass == 0 ? 0 : a.W - 1;
    g.border = false;
    if (a.r == 0) {
        g.i = id; g.j = j1; g.si = 0; g.sj = g.dj; g.len = a.W;
    } else if (a.r == 2) {
        g.i = g.i1; g.j = id; g.si = g.di; g.sj = 0; g.len = a.H;
    } else {
        g.si = g.di;
        g.sj = a.r == 1 ? g.dj : -g.dj;
        if (id < a.W) {
            g.i = g.i1; g.j = id;
        } else {
            g.i = g.i1 + g.di * (id - a.W + 1);
            g.j = a.r == 1 ? j1 : (a.W - 1 - j1);
            g.border = true;
        }
        const int rows_left = g.di > 0 ? a.H - g.i : g.i + 1;
        const int cols_left = g.sj > 0 ? a.W - g.j : g.j + 1;
        g.len = min(rows_left, cols_left);
    }
    return g;
}

// P2 of path r at pixel (i, j): intensities from the flat stream (RSGM/StereoSGM_SSE.hpp:238-243)
__device__ __forceinline__ int path_p2(const SgmArgs &a, const LineGeom &g, const uint8_t *img, int i, int j)
{
    const int il = (i == g.i1 + g.di) ? i : i - g.di;
    long q;
    if (a.r == 0) q = (long)i * a.W + j - g.dj;
    else if (a.r == 1) q = (long)il * a.W + j - g.dj;
    else if (a.r == 2) q = (long)il * a.W + j;
    else q = (long)il * a.W + j + g.dj;
    const long n = (long)a.W * a.H;
    q = q < 0 ? 0 : (q >= n ? n - 1 : q);      // never taken for H >= 3; keeps degenerate shapes in bounds
    return adapt_p2(a.p, img[(long)i * a.W + j], img[q]);
}

// ------------------------------------------------------------------------------------------------------------
// fast instantiation: uint8 costs, packed u16x2 arithmetic
// ------------------------------------------------------------------------------------------------------------
#define BIG16 0x3FFFu
#define BIG2 0x3FFF3FFFu

template <int NW, bool PAD, bool STORE>
__global__ void __launch_bounds__(128) sgm_path_fast_kernel(const uint8_t *__restrict__ img_all, const uint8_t *__restrict__ dsi_all,
                                                            uint16_t *__restrict__ S_all, SgmArgs a, long total_lines)
{
    const long gl = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (gl >= total_lines) return;
    const int lane = threadIdx.x & 31;
    const long f = gl / a.lines;
    const int id = (int)(gl % a.lines);
    const LineGeom g = line_geom(a, id);
    const long npx = (long)a.W * a.H;
    const uint8_t *img = img_all + f * npx;
    const uint8_t *dsi = dsi_all + f * npx * a.D;
    uint16_t *S = S_all + f * npx * a.D;
    const int d0 = 2 * NW * lane;

    uint32_t vm[NW];                       // per-word valid mask (PAD only)
#pragma unroll
    for (int k = 0; k < NW; k++) {
        const int d = d0 + 2 * k;
        vm[k] = (d < a.D ? 0x0000FFFFu : 0u) | (d + 1 < a.D ? 0xFFFF0000u : 0u);
    }
    const bool lane_on = d0 < a.D;

    uint32_t w[NW];                        // L of the previous pixel on the line
    uint32_t mprev = 0;
    const uint32_t P1x2 = (uint32_t)a.p.P1 * 0x10001u;

    // software prefetch of the next pixel's costs, S words and P2
    uint32_t c_next[NW], s_next[NW];
    int p2_next = 0;
    auto load_px = [&](int t, uint32_t (&c)[NW], uint32_t (&s)[NW], int &p2) {
        const int i = g.i + t * g.si, j = g.j + t * g.sj;
        const long px = (long)i * a.W + j;
#pragma unroll
        for (int k = 0; k < NW; k++) {
            const int d = d0 + 2 * k;
            uint32_t cv = 0;
            if (!PAD || d < a.D) cv = *reinterpret_cast<const uint16_t *>(dsi + px * a.D + d);
            c[k] = __byte_perm(cv, 0, 0x4140);            // two uint8 costs -> u16x2
            if (!STORE) s[k] = (!PAD || d < a.D) ? *reinterpret_cast<const uint32_t *>(S + px * a.D + d) : 0u;
        }
        p2 = (t > 0 || g.border) ? path_p2(a, g, img, i, j) : 0;
    };
    load_px(0, c_next, s_next, p2_next);

    for (int t = 0; t < g.len; t++) {
        uint32_t c[NW], s[NW];
#pragma unroll
        for (int k = 0; k < NW; k++) { c[k] = c_next[k]; s[k] = s_next[k]; }
        const int p2 = p2_next;
        if (t + 1 < g.len) load_px(t + 1, c_next, s_next, p2_next);

        uint32_t nw[NW];
        bool add_to_s = true;
        if (t == 0 && !g.border) {
            // first pixel of the line: L = C.  Only r0 contributes it to S (first row of a pass sums r0 only).
#pragma unroll
            for (int k = 0; k < NW; k++) nw[k] = c[k];
            add_to_s = (a.r == 0);
        } else if (t == 0) {
            // enters through the side border: min(65535, 65535+P1, 0 + P2) - 0 = P2
            const uint32_t p2x2 = (uint32_t)p2 * 0x10001u;
#pragma unroll
            for (int k = 0; k < NW; k++) nw[k] = c[k] + p2x2;
        } else {
            uint32_t up = __shfl_up_sync(0xFFFFFFFFu, w[NW - 1], 1);
            uint32_t dn = __shfl_down_sync(0xFFFFFFFFu, w[0], 1);
            if (lane == 0) up = BIG2;
            if (lane == 31) dn = BIG2;
            uint32_t ext[NW + 2];
            ext[0] = up;
#pragma unroll
            for (int k = 0; k < NW; k++) ext[k + 1] = w[k];
            ext[NW + 1] = dn;
            uint32_t p[NW + 1];
#pragma unroll
            for (int k = 0; k <= NW; k++) p[k] = __byte_perm(ext[k], ext[k + 1], 0x5432);   // (hi(ext[k]), lo(ext[k+1]))
            const uint32_t mP2 = (mprev + (uint32_t)p2) * 0x10001u;
            const uint32_t mx2 = mprev * 0x10001u;
#pragma unroll
            for (int k = 0; k < NW; k++) {
                uint32_t tmin = __vminu2(p[k], p[k + 1]);               // min(L[d-1], L[d+1])
                tmin = __viaddmin_u16x2(tmin, P1x2, w[k]);              // min(. + P1, L[d])
                tmin = __vminu2(tmin, mP2);                             // min(., minL + P2)
                nw[k] = tmin + c[k] - mx2;                              // every candidate >= minL: no borrow
            }
        }
        if (PAD) {
#pragma unroll
            for (int k = 0; k < NW; k++) nw[k] = (nw[k] & vm[k]) | (BIG2 & ~vm[k]);
        }
        // minimum over all disparities
        uint32_t mm = nw[0];
#pragma unroll
        for (int k = 1; k < NW; k++) mm = __vminu2(mm, nw[k]);
        mm = min(mm & 0xFFFFu, mm >> 16);
        mprev = __reduce_min_sync(0xFFFFFFFFu, mm);
#pragma unroll
        for (int k = 0; k < NW; k++) w[k] = nw[k];

        if (add_to_s && lane_on) {
            const int i = g.i + t * g.si, j = g.j + t * g.sj;
            uint16_t *sp = S + ((long)i * a.W + j) * a.D;
#pragma unroll
            for (int k = 0; k < NW; k++) {
                const int d = d0 + 2 * k;
                if (!PAD || d < a.D) *reinterpret_cast<uint32_t *>(sp + d) = STORE ? nw[k] : s[k] + nw[k];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// generic instantiation: uint16 (CT = uint16_t) or uint8 costs, arbitrary parameters, explicit uint16 saturation (SSE adds/subs
// semantics)
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t sat16(uint32_t v) { return v > 65535u ? 65535u : v; }

template <int NW, typename CT>
__global__ void __launch_bounds__(128) sgm_path_generic_kernel(const uint8_t *__restrict__ img_all, const CT *__restrict__ dsi_all,
                                                               uint16_t *__restrict__ S_all, SgmArgs a, long total_lines)
{
    constexpr int ND = 2 * NW;
    const long gl = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (gl >= total_lines) return;
    const int lane = threadIdx.x & 31;
    const long f = gl / a.lines;
    const int id = (int)(gl % a.lines);
    const LineGeom g = line_geom(a, id);
    const long npx = (long)a.W * a.H;
    const uint8_t *img = img_all + f * npx;
    const CT *dsi = dsi_all + f * npx * a.D;
    uint16_t *S = S_all + f * npx * a.D;
    const int d0 = ND * lane;
    const bool store = (a.r == 0 && a.pass == 0);

    uint32_t L[ND];
    uint32_t mprev = 0;
    for (int t = 0; t < g.len; t++) {
        const int i = g.i + t * g.si, j = g.j + t * g.sj;
        const long px = (long)i * a.W + j;
        uint32_t c[ND];
#pragma unroll
        for (int k = 0; k < ND; k++) c[k] = (d0 + k < a.D) ? dsi[px * a.D + d0 + k] : 65535u;
        uint32_t nl[ND];
        bool add_to_s = true;
        if (t == 0 && !g.border) {
#pragma unroll
            for (int k = 0; k < ND; k++) {
                uint32_t cv = c[k];
                if (i == g.i1 && cv == 255u) cv = 12u;          // first line only (:120,:134,:157); unreachable for census
                nl[k] = cv;
            }
            add_to_s = (a.r == 0);
        } else {
            uint32_t up, dn;
            {
                uint32_t u = __shfl_up_sync(0xFFFFFFFFu, L[ND - 1], 1);
                uint32_t v = __shfl_down_sync(0xFFFFFFFFu, L[0], 1);
                up = lane == 0 ? 65535u : u;
                dn = lane == 31 ? 65535u : v;
            }
            const bool from_border = (t == 0);
            const int p2 = path_p2(a, g, img, i, j);
            const uint32_t mp = from_border ? 0u : mprev;
            const uint32_t cur_p2 = sat16((uint32_t)p2 + mp);       // _mm_adds_epu16(varP2, minL)
#pragma unroll
            for (int k = 0; k < ND; k++) {
                uint32_t lm, ld, lp;
                if (from_border) { lm = ld = lp = 65535u; }
                else {
                    ld = L[k];
                    lm = k == 0 ? up : L[k - 1];
                    lp = k == ND - 1 ? dn : L[k + 1];
                }
                uint32_t m = min(min(ld, sat16(lm + (uint32_t)a.p.P1)), min(sat16(lp + (uint32_t)a.p.P1), cur_p2));
                m = m > mp ? m - mp : 0u;                           // _mm_subs_epu16
                uint32_t cv = c[k];
                if (a.r == 0 && i == g.i1 && cv == 255u) cv = 12u;  // r0 on the first line runs the scalar code (:157)
                nl[k] = sat16(cv + m);
            }
        }
        uint32_t mm = 65535u;
#pragma unroll
        for (int k = 0; k < ND; k++) {
            if (d0 + k >= a.D) nl[k] = 65535u;                      // padded disparities behave like the d = D slot
            mm = min(mm, nl[k]);
            L[k] = nl[k];
        }
        mprev = __reduce_min_sync(0xFFFFFFFFu, mm);
        if (add_to_s) {
            const bool wrap = (a.pass == 1 && i == g.i1);           // `+=` on uint16 (:143,:198)
#pragma unroll
            for (int k = 0; k < ND; k++) {
                if (d0 + k < a.D) {
                    uint16_t *sp = S + px * a.D + d0 + k;
                    if (store) *sp = (uint16_t)nl[k];
                    else if (wrap) *sp = (uint16_t)(*sp + nl[k]);
                    else *sp = (uint16_t)sat16((uint32_t)*sp + nl[k]);
                }
            }
        }
    }
}

static int lines_for(int r, int W, int H) { return r == 0 ? H : (r == 2 ? W : W + H - 1); }

template <int NW>
static int run_fast(const uint8_t *img, const uint8_t *dsi, uint16_t *S, SgmArgs a, int n, cudaStream_t st)
{
    const bool pad = (a.D != 64 * NW);
    for (int pass = 0; pass < 2; pass++)
        for (int r = 0; r < 4; r++) {
            a.r = r; a.pass = pass; a.lines = lines_for(r, a.W, a.H);
            const long total = (long)n * a.lines;
            const int blocks = cdiv(total * 32, 128);
            const bool store = (r == 0 && pass == 0);
            if (store) {
                if (pad) sgm_path_fast_kernel<NW, true, true><<<blocks, 128, 0, st>>>(img, dsi, S, a, total);
                else sgm_path_fast_kernel<NW, false, true><<<blocks, 128, 0, st>>>(img, dsi, S, a, total);
            } else {
                if (pad) sgm_path_fast_kernel<NW, true, false><<<blocks, 128, 0, st>>>(img, dsi, S, a, total);
                else sgm_path_fast_kernel<NW, false, false><<<blocks, 128, 0, st>>>(img, dsi, S, a, total);
            }
            VPP_LAUNCH_CHECK("sgm_path_fast_kernel");
        }
    return VPPB200_OK;
}

int launch_aggregate_fast(const uint8_t *img, const uint8_t *dsi, uint16_t *S, int W, int H, int D, const SgmParams &p, int n,
                          cudaStream_t st)
{
    SgmArgs a;
    a.W = W; a.H = H; a.D = D; a.p = p;
    a.r = 0; a.pass = 0; a.lines = 0;
    switch ((D + 63) / 64) {
        case 1: return run_fast<1>(img, dsi, S, a, n, st);
        case 2: return run_fast<2>(img, dsi, S, a, n, st);
        case 3: return run_fast<3>(img, dsi, S, a, n, st);
        default: return run_fast<4>(img, dsi, S, a, n, st);
    }
}

template <int NW, typename CT>
static int run_generic(const uint8_t *img, const CT *dsi, uint16_t *S, SgmArgs a, int n, cudaStream_t st)
{
    for (int pass = 0; pass < 2; pass++)
        for (int r = 0; r < 4; r++) {
            a.r = r; a.pass = pass; a.lines = lines_for(r, a.W, a.H);
            const long total = (long)n * a.lines;
            sgm_path_generic_kernel<NW, CT><<<cdiv(total * 32, 128), 128, 0, st>>>(img, dsi, S, a, total);
            VPP_LAUNCH_CHECK("sgm_path_generic_kernel");
        }
    return VPPB200_OK;
}

template <typename CT>
static int aggregate_generic(const uint8_t *img, const CT *dsi, uint16_t *S, int W, int H, int D, const SgmParams &p, int n,
                             cudaStream_t st)
{
    SgmArgs a;
    a.W = W; a.H = H; a.D = D; a.p = p;
    a.r = 0; a.pass = 0; a.lines = 0;
    switch ((D + 63) / 64) {
        case 1: return run_generic<1>(img, dsi, S, a, n, st);
        case 2: return run_generic<2>(img, dsi, S, a, n, st);
        case 3: return run_generic<3>(img, dsi, S, a, n, st);
        default: return run_generic<4>(img, dsi, S, a, n, st);
    }
}

int launch_aggregate_generic(const uint8_t *img, const uint16_t *dsi, uint16_t *S, int W, int H, int D, int P1, int P2min,
                             float alpha, int gamma, int n, cudaStream_t st)
{
    return aggregate_generic(img, dsi, S, W, H, D, SgmParams{P1, P2min, gamma, alpha}, n, st);
}

// compute_rsgm with parameters outside the sweep domain: the uint8 cost volume in xyd order, saturating arithmetic
int launch_aggregate_generic_u8(const uint8_t *img, const uint8_t *dsi, uint16_t *S, int W, int H, int D, const SgmParams &p, int n,
                                cudaStream_t st)
{
    return aggregate_generic(img, dsi, S, W, H, D, p, n, st);
}

}  // namespace vppb200
