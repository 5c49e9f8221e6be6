// sgm.cu -- 8-path SGM aggregation on sm_100a, bit-exact with the reference's raster recursion
// (RSGM/StereoSGM_SSE.hpp:13-515 via RSGM/pyrSGM.cpp:504-637; semantics in SURVEY.md A.4).
//
// Decomposition.  The reference sweeps the image twice (pass 0 top-down/left-right, pass 1 mirrored) and updates
// four paths per pixel inside each sweep.  Every path is a family of independent 1-D recurrences, so here one WARP
// owns one path line and walks it; lane l holds disparities [2*NW*l, 2*NW*(l+1)), one per register.
//   r0 (horizontal) : one line per row, L(j1) = C
//   r2 (vertical)   : one line per column, starts on the pass's first row with L = C (not summed into S, :116-218)
//   r1, r3 (diagonal): lines that start on the first row behave like r2; lines that enter through a side column
//                     start from the border slot L = 65535, min = 0, i.e. L = C + P2 (:48-58,:69-72)
// Reproduced quirks: P2 intensities are read from the FLAT image stream (wrap across row ends); on the row right
// after a pass's first row the "previous line" is that same row (:221); row H-1 of pass 1 adds with uint16
// wrap-around (:143,:198); everything else saturates at 65535.
//
// One kernel, sgm_path_generic_kernel<NW, CT>, with any parameters and the reference's uint16 saturation: uint16 costs for the
// aggregate_SSE drop-in, the uint8 cost volume for compute_rsgm wherever the sweeps (sgm_sweep.cu) do not run -- parameters
// outside their domain, or a shape or device they cannot hold.  Inside the domain (sweep_params_supported) it gives the
// sweeps' bits: L <= Cmax + P2max <= 4095 and S <= 8 * 4095 < 65536, so neither the saturation nor the pass-1 wrap fires, and
// costs <= 240 never meet the first line's 255 -> 12 rule.
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
// uint16 (CT = uint16_t) or uint8 costs, arbitrary parameters, explicit uint16 saturation (SSE adds/subs semantics)
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

// CT = uint16_t: the aggregate_SSE drop-in; CT = uint8_t: compute_rsgm where the sweeps do not run (xyd-order cost volume)
template <typename CT>
int launch_aggregate_generic(const uint8_t *img, const CT *dsi, uint16_t *S, int W, int H, int D, const SgmParams &p, int n,
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
template int launch_aggregate_generic(const uint8_t *, const uint8_t *, uint16_t *, int, int, int, const SgmParams &, int,
                                      cudaStream_t);
template int launch_aggregate_generic(const uint8_t *, const uint16_t *, uint16_t *, int, int, int, const SgmParams &, int,
                                      cudaStream_t);

}  // namespace vppb200
