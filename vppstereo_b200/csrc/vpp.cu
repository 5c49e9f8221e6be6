// vpp.cu -- Virtual Pattern Projection on sm_100a: exact parallel restatements of the reference's sequential scans
// (vpp_core/vpp_core_opt.pyx:53-341 and the numba twin vpp_standalone.py:14-369; semantics in SURVEY.md A.1).
//
// rnd mode.  Every read that feeds a write to image row yy (of L or R) is in row yy of the same channel
// (SURVEY.md A.1.5), so the final row yy of channel j equals the ORDERED replay, over the hints of rows
// yy-n..yy+n in scan order, of the yw = yy - y slice of each patch.  One thread owns one (frame, row, channel)
// and replays its writers in order: no atomics, no races, bit-exact.  The random stream position of every draw
// is closed-form (A.1.6) from per-row prefix sums, so the pre-drawn pattern is indexed, not consumed.
//
// maxDistance mode.  The colour of a patch pixel is a fold over a 64x3 window of the CURRENT images, so hints are
// truly sequential per channel; channels are independent.  One warp owns one (frame, channel): the window samples
// are fetched 32 at a time and folded with ballot skip-ahead (only samples strictly inside the shrinking (pa,pb)
// interval can change it), lane 0 applies the blends.
//
// Blends are evaluated in the reference's mixed float32/float64 typing with truncation to uint8; this file is
// compiled with -fmad=false and uses explicit _rn intrinsics so no FMA contraction can change a truncation.
#include "common.cuh"

namespace vppb200 {

struct VppArgs {
    int W, H, C;
    int uniform, n, nax, nay, direction, discard, interpolate, arith;
    float c32, cocc32;
    double c64, cocc64;
    // adaptive patches of vpp() (vpp_standalone.py:6-11,:153-154,:334-335); both NULL = fixed (2n+1)^2 patches
    const float *filled;   // [frames][H][W] bilateral-filled hints: a patch pixel is kept iff |g - filled| < 0.1 (float64)
    const float *thr;      // [frames][nthr] ascending disparity thresholds: patch size = 1 + #{k : g >= thr[k]}
    int nthr;
    int y0, y1;            // rnd only: image rows [y0, y1) are produced (row-band split of an oversized frame), others left untouched
};

// per-hint patch radius and per-pixel keep test of the adaptive modes
__device__ __forceinline__ int patch_radius(const VppArgs &a, long f, float gv)
{
    if (!a.thr) return a.n;
    int ws = 1;
    for (int k = 0; k < a.nthr; k++) ws += gv >= a.thr[f * a.nthr + k];
    return (ws - 1) >> 1;
}
__device__ __forceinline__ bool patch_keep(const VppArgs &a, long f, float gv, int yy, int xx)
{
    if (!a.filled) return true;
    return fabs((double)gv - (double)a.filled[(f * a.H + yy) * a.W + xx]) < 0.1;
}

struct VppWs {
    uint16_t *hx;        // [n][H][W] hint columns of each row in scan order
    int *cnt;            // [n][H]   hints per row
    long long *draws;    // [n][H]   pattern draws per row and channel  (sum of in-image patch pixels)
    long long *hbase;    // [n][H]   exclusive prefix of cnt
    long long *dbase;    // [n][H]   exclusive prefix of draws
    uint32_t *hpre;      // [n][H][W] per hint (parallel to hx): in-image patch pixels of the earlier hints of its row
    uint8_t *rowflag;    // [n][H]   1 = this image row is left to the ordered-replay kernel (see vpp_rnd_rows_kernel)
};

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

static size_t vpp_ws_layout(int H, int W, int n, void *base, VppWs *ws)
{
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) { size_t o = off; off += align256(bytes); return b ? b + o : (char *)nullptr; };
    uint16_t *hx = (uint16_t *)take((size_t)n * H * W * 2);
    int *cnt = (int *)take((size_t)n * H * 4);
    long long *draws = (long long *)take((size_t)n * H * 8);
    long long *hbase = (long long *)take((size_t)n * H * 8);
    long long *dbase = (long long *)take((size_t)n * H * 8);
    uint32_t *hpre = (uint32_t *)take((size_t)n * H * W * 4);
    uint8_t *rowflag = (uint8_t *)take((size_t)n * H);
    if (ws) { ws->hx = hx; ws->cnt = cnt; ws->draws = draws; ws->hbase = hbase; ws->dbase = dbase; ws->hpre = hpre; ws->rowflag = rowflag; }
    return off;
}

// ---- per-row ordered hint compaction: one warp per (frame, row) ---------------------------------------------
__global__ void __launch_bounds__(128) vpp_compact_rows_kernel(const float *__restrict__ g, VppWs ws, int W, int H, int n_patch,
                                                               int direction, long total_rows)
{
    const long row = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= total_rows) return;
    const int lane = threadIdx.x & 31;
    const int y = (int)(row % H);
    const float *grow = g + row * W;
    uint16_t *out = ws.hx + row * W;
    const int ny = min(y + n_patch, H - 1) - max(y - n_patch, 0) + 1;
    int count = 0;
    long long draws = 0;
    for (int base = 0; base < W; base += 32) {
        const int s = base + lane;                       // position in scan order
        const int x = direction != 0 ? s : W - 1 - s;
        const bool hit = s < W && grow[x] > 0.0f;
        const unsigned m = __ballot_sync(0xFFFFFFFFu, hit);
        const int nx1 = hit ? (min(x + n_patch, W - 1) - max(x - n_patch, 0) + 1) : 0;
        int incl = nx1;                                  // inclusive warp scan of the patch widths
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += t;
        }
        if (hit) {
            const int slot = count + __popc(m & ((1u << lane) - 1u));
            out[slot] = (uint16_t)x;
            ws.hpre[row * W + slot] = (uint32_t)(draws + (long long)(incl - nx1) * ny);
        }
        draws += (long long)__shfl_sync(0xFFFFFFFFu, incl, 31) * ny;
        count += __popc(m);
    }
    if (lane == 0) { ws.cnt[row] = count; ws.draws[row] = draws; }
}

// exclusive prefix over the rows of each frame: one warp per frame, 32 rows per step
__global__ void __launch_bounds__(128) vpp_scan_rows_kernel(VppWs ws, int H, int n, int32_t *n_hints_out)
{
    const int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (f >= n) return;
    const int lane = threadIdx.x & 31;
    long long hb = 0, db = 0;
    for (int y0 = 0; y0 < H; y0 += 32) {
        const int y = y0 + lane;
        const long r = (long)f * H + y;
        const long long c = y < H ? ws.cnt[r] : 0, d = y < H ? ws.draws[r] : 0;
        long long ci = c, di = d;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long tc = __shfl_up_sync(0xFFFFFFFFu, ci, o), td = __shfl_up_sync(0xFFFFFFFFu, di, o);
            if (lane >= o) { ci += tc; di += td; }
        }
        if (y < H) { ws.hbase[r] = hb + ci - c; ws.dbase[r] = db + di - d; }
        hb += __shfl_sync(0xFFFFFFFFu, ci, 31); db += __shfl_sync(0xFFFFFFFFu, di, 31);
    }
    if (n_hints_out && lane == 0) n_hints_out[f] = (int32_t)hb;
}

// ---- the blend of one patch pixel (vpp_core_opt.pyx:104-124 / :315-335; vpp_standalone.py:342-363 / :206-226) -----
__device__ __forceinline__ uint8_t tr8(double v) { return (uint8_t)(int)v; }     // truncation; values are in [0,256)

struct Splat {
    const VppArgs &a;
    uint8_t *lrow, *rrow;      // row pointers at channel j (pixel stride = C)
    __device__ __forceinline__ uint8_t getL(int x) const { return lrow[(long)x * a.C]; }
    __device__ __forceinline__ void setL(int x, uint8_t v) const { lrow[(long)x * a.C] = v; }
    __device__ __forceinline__ uint8_t getR(int x) const { return rrow[(long)(x < 0 ? x + a.W : x) * a.C]; }  // negative index wraps
    __device__ __forceinline__ void setR(int x, uint8_t v) const { rrow[(long)(x < 0 ? x + a.W : x) * a.C] = v; }
};

// pv: pattern value (rnd: the drawn uint8; maxDistance: (pa+pb)/2 as double)
template <bool RND, class S>
__device__ __forceinline__ void splat_pixel(const S &s, double pv, int xl, int x0, int x1, int xr, bool occluded,
                                            float b32, double b64)
{
    const VppArgs &a = s.a;
    const int W = a.W;
    // colour term and (1 - c) in the reference's typing
    auto colour = [&](bool occ) -> double {
        if (a.arith == 0) {
            const float c = occ ? a.cocc32 : a.c32;
            if (RND) return (double)__fmul_rn((float)pv, c);          // uint8 * float -> float
            return __dmul_rn(pv, (double)c);                          // double * float -> double
        }
        return __dmul_rn(pv, occ ? a.cocc64 : a.c64);
    };
    auto omc = [&](bool occ) -> double {
        if (a.arith == 0) return __dsub_rn(1.0, (double)(occ ? a.cocc32 : a.c32));
        return __dsub_rn(1.0, occ ? a.cocc64 : a.c64);
    };
    const double b = a.arith == 0 ? (double)b32 : b64;
    const double omb = __dsub_rn(1.0, b);
    // r * b: uint8 * float32 -> float32 in the Cython build, double in numba
    auto r_times_b = [&](uint8_t r) -> double {
        if (a.arith == 0) return (double)__fmul_rn((float)r, b32);
        return __dmul_rn((double)r, b64);
    };
    auto blend = [&](double rc, uint8_t old, double om) -> double { return __dadd_rn(rc, __dmul_rn((double)old, om)); };

    if (0 <= x0 && x0 <= W - 1) {
        if (!occluded) {
            const double rc = colour(false), om = omc(false);
            s.setL(xl, tr8(blend(rc, s.getL(xl), om)));
            if (a.interpolate) {
                const uint8_t r0 = s.getR(x0);
                s.setR(x0, tr8(__dadd_rn(__dmul_rn(blend(rc, r0, om), omb), r_times_b(r0))));
                if (0 <= x1 && x1 <= W - 1) {
                    const uint8_t r1 = s.getR(x1);
                    s.setR(x1, tr8(__dadd_rn(__dmul_rn(blend(rc, r1, om), b), __dmul_rn((double)r1, omb))));
                }
            } else {
                s.setR(xr, tr8(blend(rc, s.getR(xr), om)));
            }
        } else if (!a.discard) {
            const double rc = colour(true), omo = omc(true), om = omc(false);
            if (a.interpolate) {
                const uint8_t r0 = s.getR(x0);
                s.setR(x0, tr8(__dadd_rn(__dmul_rn(blend(rc, r0, omo), omb), r_times_b(r0))));
                if (0 <= x1 && x1 <= W - 1) {
                    const uint8_t r1 = s.getR(x1);
                    s.setR(x1, tr8(__dadd_rn(__dmul_rn(blend(rc, r1, omo), b), __dmul_rn((double)r1, omb))));
                }
                const double mix = __dadd_rn(__dmul_rn((double)s.getR(x0), omb), r_times_b(s.getR(x1)));
                const double cc = a.arith == 0 ? (double)a.c32 : a.c64;
                s.setL(xl, tr8(__dadd_rn(__dmul_rn(mix, cc), __dmul_rn((double)s.getL(xl), om))));
            } else {
                s.setR(xr, tr8(blend(rc, s.getR(xr), omo)));
                const double rcl = a.arith == 0 ? (double)__fmul_rn((float)s.getR(xr), a.c32) : __dmul_rn((double)s.getR(xr), a.c64);
                s.setL(xl, tr8(__dadd_rn(rcl, __dmul_rn((double)s.getL(xl), om))));
            }
        }
    } else {
        s.setL(xl, tr8(blend(colour(false), s.getL(xl), omc(false))));    // left-side occlusion (pyx:123-124)
    }
}

struct HintGeom {
    int xd, xd0, xd1;
    float b32;
    double b64;
};
__device__ __forceinline__ HintGeom hint_geom(const VppArgs &a, float gv, int x)
{
    HintGeom h;
    const int d0 = (int)floorf(gv), d1 = (int)ceilf(gv);
    // (int)round(g): C round = half away from zero (pyx:82); numba round = half to even (vpp_standalone.py:304)
    const int d = a.arith == 0 ? (int)roundf(gv) : __float2int_rn(gv);
    h.xd = x - d; h.xd0 = x - d0; h.xd1 = x - d1;
    h.b32 = __fsub_rn(gv, (float)d0);
    h.b64 = __dsub_rn((double)gv, (double)d0);
    return h;
}

// on-device pattern generation (pattern == NULL): counter based, value = 32-bit finaliser of (frame key, stream position
// modulo 2^32)
__device__ __forceinline__ uint32_t frame_key32(uint64_t rng_seed, long f)
{
    const uint64_t k = rng_seed ^ ((uint64_t)f * 0x9E3779B97F4A7C15ull);
    return (uint32_t)k ^ ((uint32_t)(k >> 32) * 0x85EBCA6Bu);
}
__device__ __forceinline__ uint8_t counter_pattern(uint32_t key, uint32_t idx)
{
    uint32_t h = (idx * 0x9E3779B1u) ^ key;
    h ^= h >> 16; h *= 0x85EBCA6Bu;
    h ^= h >> 13; h *= 0xC2B2AE35u;
    h ^= h >> 16;
    return (uint8_t)(h >> 24);
}

// ---- rnd: ordered replay, one thread per (frame, row yy, channel j) ------------------------------------------
__global__ void __launch_bounds__(128) vpp_rnd_replay_kernel(uint8_t *__restrict__ l, uint8_t *__restrict__ r,
                                                             const float *__restrict__ g, const uint8_t *__restrict__ g_occ,
                                                             const uint8_t *__restrict__ pattern,
                                                             const int64_t *__restrict__ pattern_offsets, uint64_t rng_seed,
                                                             VppWs ws, VppArgs a, long total, int only_flagged)
{
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int j = (int)(t % a.C);
    const int yy = (int)((t / a.C) % a.H);
    const long f = t / ((long)a.C * a.H);
    const int W = a.W, H = a.H, n = a.n;
    if (yy < a.y0 || yy >= a.y1) return;                        // outside this call's row band
    if (only_flagged && !ws.rowflag[f * H + yy]) return;        // this row was done by vpp_rnd_rows_kernel
    Splat s{a, l + ((f * H + yy) * W) * a.C + j, r + ((f * H + yy) * W) * a.C + j};
    const uint8_t *pat = pattern ? pattern + pattern_offsets[f] : nullptr;
    const long long pat_len = pattern ? pattern_offsets[f + 1] - pattern_offsets[f] : 0;
    const uint32_t frame_key = frame_key32(rng_seed, f);
    for (int y = max(0, yy - n); y <= min(H - 1, yy + n); y++) {
        const long row = f * H + y;
        const int cnt = ws.cnt[row];
        const uint16_t *hx = ws.hx + row * W;
        const int ylo = max(y - n, 0);                        // first in-image patch row
        const int ny = min(y + n, H - 1) - ylo + 1;
        const int rows_before = yy - ylo;                     // in-image patch rows above the slice
        long long draw_prefix = ws.dbase[row];                // draws (per channel) of earlier hints
        const long long hint_prefix = ws.hbase[row];
        for (int k = 0; k < cnt; k++) {
            const int x = hx[k];
            const float gv = g[row * W + x];
            const bool occ = g_occ[row * W + x] != 0;
            const HintGeom hg = hint_geom(a, gv, x);
            const int xlo = max(x - n, 0), xhi = min(x + n, W - 1);
            const int nx = xhi - xlo + 1;
            const long long inb = (long long)nx * ny;
            // stream index of the first pixel of my slice (SURVEY.md A.1.6)
            long long idx = a.uniform ? (long long)a.C * (hint_prefix + k) + j
                                      : (long long)a.C * draw_prefix + (long long)j * inb + (long long)rows_before * nx;
            for (int xx = xlo; xx <= xhi; xx++) {
                const int xw = xx - x;
                const uint8_t rv = pat ? ((idx >= 0 && idx < pat_len) ? pat[idx] : 0) : counter_pattern(frame_key, (uint32_t)idx);
                if (!a.uniform) idx++;
                splat_pixel<true>(s, (double)rv, xx, hg.xd0 + xw, hg.xd1 + xw, hg.xd + xw, occ, hg.b32, hg.b64);
            }
            draw_prefix += inb;
        }
    }
}

// ---- rnd: per-pixel replay, one CTA per (frame, image row yy) -------------------------------------------------
// Finer than the per-row replay above and still exact: when no hint of the rows yy-n..yy+n is occluded-and-kept, every
// blend reads only the pixel it writes (SURVEY.md A.1.1-A.1.4), so the final value of a pixel is the fold, in scan order,
// of the blends that target it.  The CTA (1) stages the hints of its 2n+1 source rows, (2) turns every (hint, xw) into
// up to three write records -- left pixel x+xw, right pixels x-d0+xw and x-d1+xw -- and bins them by target pixel in
// shared memory (count, exclusive scan, fill), (3) lets one thread per target pixel sort its few records by scan order
// and replay them for all channels.  Thousands of independent pixels per row instead of one thread per row.
// Rows it cannot take (an occluded hint that is not discarded: its left blend reads the right image; more hints or
// records than the shared-memory bins hold; patches wider than 15) are flagged and left to vpp_rnd_replay_kernel.
struct RowsCfg { int cap_rec, cap_hint; };
static constexpr int VR_NT = 512;

// the write records of one (hint, xw): calls emit(target, type) with target in [0, W) = left pixel, [W, 2W) = right pixel;
// type 0 / 1 = interpolated right blend at x0 / x1, 2 = plain blend
template <typename F>
__device__ __forceinline__ void vr_records(const VppArgs &a, int x, float gv, bool occ, int xw, F emit)
{
    const int W = a.W;
    const HintGeom hg = hint_geom(a, gv, x);
    const int x0 = hg.xd0 + xw, x1 = hg.xd1 + xw;
    if (0 <= x0 && x0 <= W - 1) {
        if (occ) return;                                   // occluded and discarded (kept ones never get here)
        emit(x + xw, 2);
        if (a.interpolate) {
            emit(W + x0, 0);
            if (0 <= x1 && x1 <= W - 1) emit(W + x1, 1);
        } else {
            const int xr = hg.xd + xw;
            emit(W + (xr < 0 ? xr + W : xr), 2);
        }
    } else {
        emit(x + xw, 2);                                   // left-side occlusion (pyx:123-124)
    }
}

__global__ void __launch_bounds__(VR_NT) vpp_rnd_rows_kernel(uint8_t *__restrict__ l, uint8_t *__restrict__ r,
                                                             const float *__restrict__ g, const uint8_t *__restrict__ g_occ,
                                                             const uint8_t *__restrict__ pattern,
                                                             const int64_t *__restrict__ pattern_offsets, uint64_t rng_seed,
                                                             VppWs ws, VppArgs a, RowsCfg cfg)
{
    extern __shared__ __align__(16) uint8_t vsm[];
    const int W = a.W, H = a.H, n = a.n, C = a.C;
    const int tid = threadIdx.x;
    const long fr = blockIdx.x;                           // f * H + yy
    const int yy = (int)(fr % H);
    const long f = fr / H;
    if (yy < a.y0 || yy >= a.y1) return;                  // outside this call's row band (the replay kernel skips it too)
    const int ylo_row = max(0, yy - n), yhi_row = min(H - 1, yy + n);
    const int nrows = yhi_row - ylo_row + 1;
    __shared__ int rowstart[17];
    __shared__ long long rowdb[16], rowhb[16];
    __shared__ int s_flag0, s_flag, s_flag2, s_total;      // one flag per decision point: no thread re-reads a flag others still set
    if (tid == 0) {
        int acc = 0;
        for (int i = 0; i < nrows && i < 16; i++) {
            const long row = f * H + ylo_row + i;
            rowstart[i] = acc; acc += ws.cnt[row];
            rowdb[i] = ws.dbase[row]; rowhb[i] = ws.hbase[row];
        }
        for (int i = min(nrows, 16); i < 17; i++) rowstart[i] = acc;
        s_flag0 = (n > 7 || C > 4 || acc > cfg.cap_hint) ? 1 : 0;
        s_flag = 0; s_flag2 = 0;
        s_total = acc;
    }
    __syncthreads();
    const int nh = s_total;
    if (nh == 0 || s_flag0) {
        if (tid == 0) ws.rowflag[fr] = (uint8_t)(nh != 0);
        return;
    }
    // shared memory: recs[cap_rec] (64-bit), offs[2W+1], cur[2W], hint table (gv, row-relative prefix, x, flags)
    unsigned long long *recs = reinterpret_cast<unsigned long long *>(vsm);
    uint32_t *offs = reinterpret_cast<uint32_t *>(recs + cfg.cap_rec);
    uint32_t *cur = offs + (2 * W + 1);
    float *hgv = reinterpret_cast<float *>(cur + 2 * W);
    uint32_t *hpr = reinterpret_cast<uint32_t *>(hgv + cfg.cap_hint);
    uint16_t *hxx = reinterpret_cast<uint16_t *>(hpr + cfg.cap_hint);
    uint8_t *hfl = reinterpret_cast<uint8_t *>(hxx + cfg.cap_hint);        // bit 0: occluded, bits 1..4: source row index
    for (int i = tid; i < 2 * W + 1; i += VR_NT) offs[i] = 0;
    for (int h = tid; h < nh; h += VR_NT) {
        int yr = 0;
        while (yr + 1 < nrows && rowstart[yr + 1] <= h) yr++;
        const long row = f * H + ylo_row + yr;
        const int k = h - rowstart[yr];
        const int x = ws.hx[row * W + k];
        const bool occ = g_occ[row * W + x] != 0;
        hxx[h] = (uint16_t)x; hgv[h] = g[row * W + x]; hpr[h] = ws.hpre[row * W + k];
        hfl[h] = (uint8_t)((occ ? 1 : 0) | (yr << 1));
        if (occ && !a.discard) s_flag = 1;               // its left blend reads the right image: ordered replay
    }
    __syncthreads();
    if (s_flag) {
        if (tid == 0) ws.rowflag[fr] = 1;
        return;
    }
    // (2a) count the records per target
    for (int h = tid; h < nh; h += VR_NT) {
        const int x = hxx[h];
        const bool occ = hfl[h] & 1;
        for (int xw = max(-n, -x); xw <= min(n, W - 1 - x); xw++)
            vr_records(a, x, hgv[h], occ, xw, [&](int target, int) { atomicAdd(&offs[target], 1u); });
    }
    __syncthreads();
    // (2b) exclusive scan over the 2W targets: contiguous chunk per thread, block scan of the chunk sums
    {
        __shared__ uint32_t part[VR_NT];
        const int per = (2 * W + VR_NT - 1) / VR_NT;
        const int b0 = min(tid * per, 2 * W), b1 = min(b0 + per, 2 * W);
        uint32_t sum = 0;
        for (int i = b0; i < b1; i++) sum += offs[i];
        part[tid] = sum;
        __syncthreads();
        if (tid < 32) {
            uint32_t run = 0;
            for (int c0 = 0; c0 < VR_NT; c0 += 32) {
                const uint32_t v = part[c0 + tid];
                uint32_t incl = v;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                    if (tid >= o) incl += t;
                }
                part[c0 + tid] = run + incl - v;
                run += __shfl_sync(0xFFFFFFFFu, incl, 31);
            }
            if (tid == 0) { s_total = (int)run; if (run > (uint32_t)cfg.cap_rec) s_flag2 = 1; }
        }
        __syncthreads();
        uint32_t acc = part[tid];
        for (int i = b0; i < b1; i++) { const uint32_t c = offs[i]; offs[i] = acc; cur[i] = acc; acc += c; }
        if (tid == VR_NT - 1) offs[2 * W] = (uint32_t)s_total;
    }
    __syncthreads();
    if (s_flag2) {
        if (tid == 0) ws.rowflag[fr] = 1;
        return;
    }
    if (tid == 0) ws.rowflag[fr] = 0;
    // (2c) fill.  A record is 64 bits: high word = scan order (hint, xw, type) with the hint's patch size in between, low
    // word = stream position (mod 2^32) of the record's pattern value for channel 0, so the replay decodes nothing
    for (int h = tid; h < nh; h += VR_NT) {
        const int x = hxx[h], yr = hfl[h] >> 1;
        const bool occ = hfl[h] & 1;
        const int y = ylo_row + yr;
        const int ylo = max(y - n, 0), ny = min(y + n, H - 1) - ylo + 1;
        const int xlo = max(x - n, 0), nx = min(x + n, W - 1) - xlo + 1;
        const uint32_t stride = a.uniform ? 1u : (uint32_t)(nx * ny);                       // <= 225
        const uint32_t base = a.uniform ? (uint32_t)((long long)C * (rowhb[yr] + (h - rowstart[yr])))
                                        : (uint32_t)((long long)C * (rowdb[yr] + hpr[h])) + (uint32_t)((yy - ylo) * nx - xlo);
        for (int xw = max(-n, -x); xw <= min(n, W - 1 - x); xw++) {
            const uint32_t idx0 = a.uniform ? base : base + (uint32_t)(x + xw);
            vr_records(a, x, hgv[h], occ, xw, [&](int target, int type) {
                const uint32_t key = ((uint32_t)h << 14) | (stride << 6) | ((uint32_t)(xw + n) << 2) | (uint32_t)type;
                recs[atomicAdd(&cur[target], 1u)] = ((unsigned long long)key << 32) | idx0;
            });
        }
    }
    __syncthreads();
    // (3) active targets -> dense list (the `cur` bins are free again), each list sorted by scan order by one thread
    __shared__ int s_nact;
    if (tid == 0) s_nact = 0;
    __syncthreads();
    uint32_t *act = cur;
    for (int t0 = 0; t0 < 2 * W; t0 += VR_NT) {
        const int t = t0 + tid;
        const int k0 = t < 2 * W ? (int)offs[t] : 0, k1 = t < 2 * W ? (int)offs[t + 1] : 0;
        const bool on = k1 > k0;
        const unsigned m = __ballot_sync(0xFFFFFFFFu, on);
        int base = 0;
        if ((tid & 31) == 0 && m) base = atomicAdd(&s_nact, __popc(m));
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (on) {
            act[base + __popc(m & ((1u << (tid & 31)) - 1u))] = (uint32_t)t;
            for (int i = k0 + 1; i < k1; i++) {            // insertion sort: the lists are a handful of records
                const unsigned long long rec = recs[i];
                int q = i - 1;
                while (q >= k0 && recs[q] > rec) { recs[q + 1] = recs[q]; q--; }
                recs[q + 1] = rec;
            }
        }
    }
    // the colour term pv * c and the kept share old * (1 - c) only depend on a byte each: two 256-entry tables per CTA,
    // filled with the reference's typing
    __shared__ double lut_c[256], lut_o[256];
    {
        const double pv = (double)tid;
        if (tid < 256) {
            if (a.arith == 0) { lut_c[tid] = (double)__fmul_rn((float)pv, a.c32); lut_o[tid] = __dmul_rn(pv, __dsub_rn(1.0, (double)a.c32)); }
            else { lut_c[tid] = __dmul_rn(pv, a.c64); lut_o[tid] = __dmul_rn(pv, __dsub_rn(1.0, a.c64)); }
        }
    }
    __syncthreads();
    // (4) replay: one thread per (active target pixel, channel)
    const uint8_t *pat = pattern ? pattern + pattern_offsets[f] : nullptr;
    const uint32_t pat_len = pattern ? (uint32_t)min((long long)0xFFFFFFFFll, (long long)(pattern_offsets[f + 1] - pattern_offsets[f])) : 0u;
    const uint32_t frame_key = frame_key32(rng_seed, f);
    const int items = s_nact * C;
    auto replay = [&](uint32_t v, int k0, int k1, int j) -> uint32_t {
        for (int i = k0; i < k1; i++) {
            const unsigned long long rec = recs[i];
            const uint32_t key = (uint32_t)(rec >> 32);
            const uint32_t type = key & 3u;
            const uint32_t idx = (uint32_t)rec + (uint32_t)j * ((key >> 6) & 255u);
            const uint32_t rv = pat ? (idx < pat_len ? pat[idx] : 0) : counter_pattern(frame_key, idx);
            const double mix = __dadd_rn(lut_c[rv], lut_o[v]);                   // colour + old * (1 - c)
            if (type == 2) {
                v = tr8(mix);
            } else {
                const float gv = hgv[key >> 14];
                const int d0 = (int)floorf(gv);
                const float b32 = __fsub_rn(gv, (float)d0);
                const double b = a.arith == 0 ? (double)b32 : __dsub_rn((double)gv, (double)d0);
                const double omb = __dsub_rn(1.0, b);
                if (type == 0) {
                    const double rb = a.arith == 0 ? (double)__fmul_rn((float)v, b32) : __dmul_rn((double)v, b);
                    v = tr8(__dadd_rn(__dmul_rn(mix, omb), rb));
                } else {
                    v = tr8(__dadd_rn(__dmul_rn(mix, b), __dmul_rn((double)v, omb)));
                }
            }
        }
        return v;
    };
    if (C <= 4) {
        // one thread per active target pixel, all its channels: a record is decoded once for the C blends it stands for (the
        // channels differ in the pattern draw and in the pixel byte only)
        for (int it = tid; it < s_nact; it += VR_NT) {
            const int t = (int)act[it];
            const int k0 = (int)offs[t], k1 = (int)offs[t + 1];
            uint8_t *px = t < W ? l + (fr * W + t) * C : r + (fr * W + (t - W)) * C;
            uint32_t v[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int j = 0; j < 4; j++) if (j < C) v[j] = px[j];
            for (int i = k0; i < k1; i++) {
                const unsigned long long rec = recs[i];
                const uint32_t key = (uint32_t)(rec >> 32);
                const uint32_t type = key & 3u, stride = (key >> 6) & 255u;
                float b32 = 0.0f;
                double b = 0.0, omb = 1.0;
                if (type != 2) {
                    const float gv = hgv[key >> 14];
                    const int d0 = (int)floorf(gv);
                    b32 = __fsub_rn(gv, (float)d0);
                    b = a.arith == 0 ? (double)b32 : __dsub_rn((double)gv, (double)d0);
                    omb = __dsub_rn(1.0, b);
                }
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    if (j < C) {
                        const uint32_t idx = (uint32_t)rec + (uint32_t)j * stride;
                        const uint32_t rv = pat ? (idx < pat_len ? pat[idx] : 0) : counter_pattern(frame_key, idx);
                        const double mix = __dadd_rn(lut_c[rv], lut_o[v[j]]);           // colour + old * (1 - c)
                        if (type == 2) {
                            v[j] = tr8(mix);
                        } else if (type == 0) {
                            const double rb = a.arith == 0 ? (double)__fmul_rn((float)v[j], b32) : __dmul_rn((double)v[j], b);
                            v[j] = tr8(__dadd_rn(__dmul_rn(mix, omb), rb));
                        } else {
                            v[j] = tr8(__dadd_rn(__dmul_rn(mix, b), __dmul_rn((double)v[j], omb)));
                        }
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < 4; j++) if (j < C) px[j] = (uint8_t)v[j];
        }
        return;
    }
    // more than four channels: one thread per (pixel, channel) item, four pixel loads in flight per thread
    constexpr int RB = 4;
    for (int it0 = tid; it0 < items; it0 += VR_NT * RB) {
        uint8_t *px[RB];
        uint32_t v[RB];
        int k0[RB], k1[RB], jj[RB];
#pragma unroll
        for (int u = 0; u < RB; u++) {
            const int it = it0 + u * VR_NT;
            px[u] = nullptr; v[u] = 0; k0[u] = k1[u] = jj[u] = 0;
            if (it < items) {
                const int t = (int)act[it / C];
                jj[u] = it % C;
                k0[u] = (int)offs[t]; k1[u] = (int)offs[t + 1];
                px[u] = (t < W ? l + (fr * W + t) * C : r + (fr * W + (t - W)) * C) + jj[u];
                v[u] = *px[u];
            }
        }
#pragma unroll
        for (int u = 0; u < RB; u++)
            if (px[u]) *px[u] = (uint8_t)replay(v[u], k0[u], k1[u], jj[u]);
    }
}

static size_t vr_smem_bytes(int W, const RowsCfg &c)
{
    return (size_t)(4 * W + 1) * 4 + (size_t)c.cap_rec * 8 + (size_t)c.cap_hint * (4 + 4 + 2 + 1) + 16;
}

// ---- rnd with adaptive patches (per-hint radius, per-pixel keep test) -------------------------------------------
// The pattern draw of a patch pixel only happens when the pixel is kept (vpp_standalone.py:334-340), so the stream position
// of a draw is the number of kept in-image patch pixels before it.  Pass 1 counts them per hint (K_h) and scans them per
// row (hpre, draws; vpp_scan_rows_kernel then gives the per-frame prefix); pass 2 is the ordered per-row replay.
__global__ void __launch_bounds__(128) vpp_adaptive_counts_kernel(const float *__restrict__ g, VppWs ws, VppArgs a, long total_rows)
{
    const long row = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= total_rows) return;
    const int lane = threadIdx.x & 31;
    const int W = a.W, H = a.H;
    const int y = (int)(row % H);
    const long f = row / H;
    const int cnt = ws.cnt[row];
    const uint16_t *hx = ws.hx + row * W;
    long long run = 0;
    for (int base = 0; base < cnt; base += 32) {
        const int k = base + lane;
        int kept = 0;
        if (k < cnt) {
            const int x = hx[k];
            const float gv = g[row * W + x];
            const int nh = patch_radius(a, f, gv);
            for (int yy = max(y - nh, 0); yy <= min(y + nh, H - 1); yy++)
                for (int xx = max(x - nh, 0); xx <= min(x + nh, W - 1); xx++) kept += patch_keep(a, f, gv, yy, xx);
        }
        int incl = kept;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += t;
        }
        if (k < cnt) ws.hpre[row * W + k] = (uint32_t)(run + incl - kept);
        run += __shfl_sync(0xFFFFFFFFu, incl, 31);
    }
    if (lane == 0) ws.draws[row] = run;
}

__global__ void __launch_bounds__(128) vpp_rnd_adaptive_kernel(uint8_t *__restrict__ l, uint8_t *__restrict__ r,
                                                               const float *__restrict__ g, const uint8_t *__restrict__ g_occ,
                                                               const uint8_t *__restrict__ pattern,
                                                               const int64_t *__restrict__ pattern_offsets, uint64_t rng_seed,
                                                               VppWs ws, VppArgs a, long total)
{
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int j = (int)(t % a.C);
    const int yy = (int)((t / a.C) % a.H);
    const long f = t / ((long)a.C * a.H);
    const int W = a.W, H = a.H, n = a.n;
    if (yy < a.y0 || yy >= a.y1) return;                        // outside this call's row band
    Splat s{a, l + ((f * H + yy) * W) * a.C + j, r + ((f * H + yy) * W) * a.C + j};
    const uint8_t *pat = pattern ? pattern + pattern_offsets[f] : nullptr;
    const long long pat_len = pattern ? pattern_offsets[f + 1] - pattern_offsets[f] : 0;
    const uint32_t frame_key = frame_key32(rng_seed, f);
    for (int y = max(0, yy - n); y <= min(H - 1, yy + n); y++) {
        const long row = f * H + y;
        const int cnt = ws.cnt[row];
        const uint16_t *hx = ws.hx + row * W;
        const long long draw_base = ws.dbase[row], hint_prefix = ws.hbase[row], row_draws = ws.draws[row];
        for (int k = 0; k < cnt; k++) {
            const int x = hx[k];
            const float gv = g[row * W + x];
            const int nh = patch_radius(a, f, gv);
            if (yy < y - nh || yy > y + nh) continue;
            const bool occ = g_occ[row * W + x] != 0;
            const HintGeom hg = hint_geom(a, gv, x);
            const long long pre = ws.hpre[row * W + k];
            const long long K = (k + 1 < cnt ? (long long)ws.hpre[row * W + k + 1] : row_draws) - pre;
            const int xlo = max(x - nh, 0), xhi = min(x + nh, W - 1);
            long long rank = 0;                            // kept pixels of the patch rows above the slice
            for (int py = max(y - nh, 0); py < yy; py++)
                for (int px = xlo; px <= xhi; px++) rank += patch_keep(a, f, gv, py, px);
            long long idx = a.uniform ? (long long)a.C * (hint_prefix + k) + j : (long long)a.C * (draw_base + pre) + (long long)j * K + rank;
            for (int xx = xlo; xx <= xhi; xx++) {
                if (!patch_keep(a, f, gv, yy, xx)) continue;
                const int xw = xx - x;
                const uint8_t rv = pat ? ((idx >= 0 && idx < pat_len) ? pat[idx] : 0) : counter_pattern(frame_key, (uint32_t)idx);
                if (!a.uniform) idx++;
                splat_pixel<true>(s, (double)rv, xx, hg.xd0 + xw, hg.xd1 + xw, hg.xd + xw, occ, hg.b32, hg.b64);
            }
        }
    }
}

// ---- _bilateral_filling (vpp_standalone.py:371-394): one thread per TARGET pixel ---------------------------------
// The reference scatters from every hint, in raster order, to the pixels of its patch and keeps the largest weight (first
// one on ties, cmap stored as float32 and compared as float64).  Gathering the candidate hints of one target in the same
// raster order reproduces it exactly.  weights[((yw+n)*(2n+1) + (xw+n))*256 + |di|] = exp(-(r^2/(2 o_xy^2) + di^2/(2 o_i^2)))
// is tabulated by the caller with the host's libm (the function numba calls), so no device exp() is involved.
__global__ void __launch_bounds__(256) bilateral_filling_kernel(const float *__restrict__ dmap, const uint8_t *__restrict__ gray,
                                                                float *__restrict__ out, int W, int H, int n,
                                                                const double *__restrict__ weights, double th, long total)
{
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int tx = (int)(t % W), ty = (int)((t / W) % H);
    const long fo = (t / ((long)W * H)) * (long)W * H;
    const int it = gray[t];
    float cmap = 0.0f, aug = dmap[t];
    const int side = 2 * n + 1;
    for (int y = max(ty - n, 0); y <= min(ty + n, H - 1); y++)
        for (int x = max(tx - n, 0); x <= min(tx + n, W - 1); x++) {
            const float d = dmap[fo + (long)y * W + x];
            if (!(d > 0.0f)) continue;
            const int di = abs(it - (int)gray[fo + (long)y * W + x]);
            const double w = weights[(((ty - y) + n) * side + ((tx - x) + n)) * 256 + di];
            if ((double)cmap < w) { cmap = (float)w; aug = d; }
        }
    out[t] = ((double)cmap > th) ? aug : 0.0f;
}

// ---- gray context of _bilateral_filling (vpp_standalone.py:415-417): cv2.cvtColor(BGR2GRAY) in OpenCV's 15-bit fixed point,
// otherwise the first channel (np.squeeze of a one-channel image).  One thread = one pixel.
__global__ void __launch_bounds__(256) bgr2gray_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ gray, int C, long total)
{
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const uint8_t *p = src + t * C;
    gray[t] = C == 3 ? (uint8_t)((p[0] * 3735u + p[1] * 19235u + p[2] * 9798u + 16384u) >> 15) : p[0];
}

// ---- distance-based patch size (vpp_standalone.py:6-9) without a host round trip ----------------------------------------
// size(d) = round(float64(ratio32(d)) ** (1/gamma) * (wsize-1) + 1) is non-decreasing in the float32 ratio, and ratio32 is
// non-decreasing in d, so size(d) >= k  <=>  ratio32(d) >= R_k, R_k = the smallest float32 ratio in [0, 1] of size >= k (host
// table, the only pow()).  One CTA per frame: dmin / dmax over the hints (float min / max: exact in any order), then one thread
// per step bisects the float32 bit patterns of [dmin, dmax] as _patch_thresholds does.
__device__ __forceinline__ float patch_ratio32(float d, float dmin, float span) { return __fdiv_rn(__fsub_rn(d, dmin), span); }

__global__ void __launch_bounds__(1024) distance_patch_thresholds_kernel(const float *__restrict__ g, long hw,
                                                                         const float *__restrict__ ratio_steps, int nthr,
                                                                         float *__restrict__ thr, int32_t *__restrict__ status)
{
    const float *gf = g + (long)blockIdx.x * hw;
    float lo = INFINITY, hi = -INFINITY;
    // scalar head up to 16-byte alignment, float4 body (4 loads in flight per thread), scalar tail
    const long head = min(hw, (long)((16 - ((uintptr_t)gf & 15)) & 15) / 4);
    const long n4 = (hw - head) / 4;
    auto take = [&](float v) { if (v > 0.0f) { lo = fminf(lo, v); hi = fmaxf(hi, v); } };
    for (long i = threadIdx.x; i < head; i += blockDim.x) take(gf[i]);
    const float4 *g4 = reinterpret_cast<const float4 *>(gf + head);
    for (long i = threadIdx.x; i < n4; i += 4L * blockDim.x) {
        float4 v[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const long q = i + (long)j * blockDim.x;
            v[j] = q < n4 ? __ldg(g4 + q) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
#pragma unroll
        for (int j = 0; j < 4; j++) { take(v[j].x); take(v[j].y); take(v[j].z); take(v[j].w); }
    }
    for (long i = head + 4 * n4 + threadIdx.x; i < hw; i += blockDim.x) take(gf[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xFFFFFFFFu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xFFFFFFFFu, hi, o));
    }
    __shared__ float s_lo[32], s_hi[32];
    const int warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    if ((threadIdx.x & 31) == 0) { s_lo[warp] = lo; s_hi[warp] = hi; }
    __syncthreads();
    lo = s_lo[0]; hi = s_hi[0];
    for (int w = 1; w < nwarps; w++) { lo = fminf(lo, s_lo[w]); hi = fmaxf(hi, s_hi[w]); }
    // no hints: the steps are never read; dmin == dmax: the reference raises ZeroDivisionError -- patch size 1 and status set
    const bool degenerate = lo == hi;
    if (degenerate && threadIdx.x == 0 && status) status[blockIdx.x] = 1;
    const float span = __fsub_rn(hi, lo);
    for (int k = threadIdx.x; k < nthr; k += blockDim.x) {
        const float R = ratio_steps[k];
        float out = INFINITY;
        if (!(lo > hi) && !degenerate && patch_ratio32(hi, lo, span) >= R) {
            uint32_t a = __float_as_uint(lo), b = __float_as_uint(hi);      // positive floats: bit order = value order
            if (patch_ratio32(lo, lo, span) >= R) b = a;
            while (a < b) {                                                  // invariant: ratio32(b) >= R
                const uint32_t mid = a + (b - a) / 2;
                if (patch_ratio32(__uint_as_float(mid), lo, span) >= R) b = mid;
                else a = mid + 1;
            }
            out = __uint_as_float(b);
        }
        thr[(long)blockIdx.x * nthr + k] = out;
    }
}

// ---- maxDistance: one warp per (frame, channel), sequential over hints ------------------------------------------
// fold of the ordered window samples into (pa, pb)  (pyx:216-313): lane p of a chunk holds window position
// chunk*32+p with up to two samples (left first, then right).
struct MaxDistState { int pa, pb, zeros; };

__device__ __forceinline__ void fold_chunk(MaxDistState &st, bool has_l, int vl, bool has_r, int vr, int lane)
{
    // book-keeping of zero samples (n_bins); which samples count is decided by the caller through has_* flags
    // ordered fold with skip-ahead: order index = 2*lane + side
    int done = -1;                                             // last consumed order index
    while (true) {
        const bool pl = has_l && (2 * lane > done) && vl > st.pa && vl < st.pb;
        const bool pr = has_r && (2 * lane + 1 > done) && vr > st.pa && vr < st.pb;
        const unsigned bl = __ballot_sync(0xFFFFFFFFu, pl), br = __ballot_sync(0xFFFFFFFFu, pr);
        const unsigned any = bl | br;
        if (!any) break;
        const int src = __ffs(any) - 1;
        const bool left_first = (bl >> src) & 1u;
        const int v = __shfl_sync(0xFFFFFFFFu, left_first ? vl : vr, src);
        done = 2 * src + (left_first ? 0 : 1);
        if (v - st.pa > st.pb - v) st.pb = v;
        else if (v - st.pa < st.pb - v) st.pa = v;
    }
}

// window sample sources: the images themselves (serial kernel) or the per-hint shared-memory region (wavefront kernel)
struct MdGlobalSrc {
    const uint8_t *limg, *rimg;       // frame base + channel j
    int W, C;
    __device__ __forceinline__ int L(int yy, int xx) const { return limg[((long)yy * W + xx) * C]; }
    __device__ __forceinline__ int R(int yy, int xx, int xr) const { (void)xx; return rimg[((long)yy * W + xr) * C]; }
};
struct MdRegionSrc {
    const uint8_t *sL, *sR;           // [RH][RW] samples of L at (oy+ry, ox+cx) and of R at (oy+ry, ox+cx-shift)
    int oy, ox, RW;
    __device__ __forceinline__ int L(int yy, int xx) const { return sL[(yy - oy) * RW + (xx - ox)]; }
    __device__ __forceinline__ int R(int yy, int xx, int xr) const { (void)xr; return sR[(yy - oy) * RW + (xx - ox)]; }
};

template <class Src>
__device__ __forceinline__ double max_dist_colour(const VppArgs &a, const Src &src, int cy, int cx, int shift,
                                                  bool occ, bool uniform_branch, int lane)
{
    const int W = a.W, H = a.H;
    const int wx = 2 * a.nax + 1, wy = 2 * a.nay + 1, npos = wx * wy;
    MaxDistState st{0, 255, 0};
    // Cython's uniform branch only counts samples that pass the range test (pyx:235-237,:248-250); a zero sample never
    // does, so n_bins cannot reach 0 there.  Everywhere else every sample is counted.
    const bool count_all = !(a.arith == 0 && uniform_branch);
    for (int base = 0; base < npos; base += 32) {
        const int p = base + lane;
        bool has_l = false, has_r = false;
        int vl = 0, vr = 0;
        if (p < npos) {
            const int yy = cy + p / wx - a.nay, xx = cx + p % wx - a.nax;
            if (yy >= 0 && yy <= H - 1 && xx >= 0 && xx <= W - 1) {
                const int xr = xx - shift;
                has_r = (0 <= xr && xr <= W - 1);
                has_l = (!occ) || !has_r;
                if (has_l) vl = src.L(yy, xx);
                if (has_r) vr = src.R(yy, xx, xr);
            }
        }
        if (count_all)
            st.zeros += __popc(__ballot_sync(0xFFFFFFFFu, has_l && vl == 0)) + __popc(__ballot_sync(0xFFFFFFFFu, has_r && vr == 0));
        fold_chunk(st, has_l, vl, has_r, vr, lane);
    }
    if (count_all && st.zeros == 256) {
        // n_bins == 0 (exactly 256 zero samples): pa = pb = first index of the minimum bin count (pyx:252-260,:305-313).
        // Rare; recount the window per candidate value.  Cython bins are int, numba bins are uint8 (wrap at 256).
        int best_k = 0, best_v = 0x7FFFFFFF;
        for (int k0 = 0; k0 < 256; k0 += 32) {
            const int k = k0 + lane;
            int cntk = 0;
            for (int p = 0; p < npos; p++) {
                const int yy = cy + p / wx - a.nay, xx = cx + p % wx - a.nax;
                if (yy < 0 || yy > H - 1 || xx < 0 || xx > W - 1) continue;
                const int xr = xx - shift;
                const bool hr = (0 <= xr && xr <= W - 1);
                if (((!occ) || !hr) && src.L(yy, xx) == k) cntk++;
                if (hr && src.R(yy, xx, xr) == k) cntk++;
            }
            if (a.arith == 1) cntk &= 255;
            // warp arg-min, first index on ties
            int key_v = cntk, key_k = k;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const int ov = __shfl_xor_sync(0xFFFFFFFFu, key_v, o), ok = __shfl_xor_sync(0xFFFFFFFFu, key_k, o);
                if (ov < key_v || (ov == key_v && ok < key_k)) { key_v = ov; key_k = ok; }
            }
            if (key_v < best_v) { best_v = key_v; best_k = key_k; }
        }
        st.pa = st.pb = best_k;
    }
    return (double)(st.pa + st.pb) / 2.0;
}

__global__ void __launch_bounds__(32) vpp_max_dist_kernel(uint8_t *l, uint8_t *r, const float *__restrict__ g,
                                                          const uint8_t *__restrict__ g_occ, VppWs ws, VppArgs a, int total)
{
    const int unit = blockIdx.x;                      // one warp per block
    if (unit >= total) return;
    const int lane = threadIdx.x;
    const int j = unit % a.C;
    const long f = unit / a.C;
    const int W = a.W, H = a.H, n = a.n;
    uint8_t *limg = l + f * (long)H * W * a.C, *rimg = r + f * (long)H * W * a.C;
    const MdGlobalSrc src{limg + j, rimg + j, W, a.C};
    for (int y = 0; y < H; y++) {
        const long row = f * H + y;
        const int cnt = ws.cnt[row];
        const uint16_t *hx = ws.hx + row * W;
        for (int k = 0; k < cnt; k++) {
            const int x = hx[k];
            const float gv = g[row * W + x];
            const bool occ = g_occ[row * W + x] != 0;
            const HintGeom hg = hint_geom(a, gv, x);
            const int nh = patch_radius(a, f, gv);
            double pv = 0.0;
            if (a.uniform) pv = max_dist_colour(a, src, y, x, x - hg.xd, occ, true, lane);
            for (int yw = -nh; yw <= nh; yw++) {
                if (y + yw < 0 || y + yw > H - 1) continue;
                for (int xw = -nh; xw <= nh; xw++) {
                    if (x + xw < 0 || x + xw > W - 1) continue;
                    if (!patch_keep(a, f, gv, y + yw, x + xw)) continue;
                    if (!a.uniform) pv = max_dist_colour(a, src, y + yw, x + xw, x - hg.xd, occ, false, lane);
                    if (lane == 0) {
                        Splat s{a, limg + ((long)(y + yw) * W) * a.C + j, rimg + ((long)(y + yw) * W) * a.C + j};
                        splat_pixel<false>(s, pv, x + xw, hg.xd0 + xw, hg.xd1 + xw, hg.xd + xw, occ, hg.b32, hg.b64);
                    }
                    __syncwarp();                     // lane 0's stores are visible to the next window fetch
                }
            }
        }
    }
}

// The same fold for the wavefront kernel, out of the staged region: window rows are walked 32 columns at a time (no
// div/mod), the next sample that can move (pa, pb) is found with ONE warp min-reduction over keys (order << 8 | value),
// zero samples are counted per lane and summed once.  Falls back to max_dist_colour for the n_bins == 0 corner.
__device__ __forceinline__ double md_colour_region(const VppArgs &a, const MdRegionSrc &src, int cy, int cx, int shift, bool occ,
                                                   bool uniform_branch, int lane)
{
    const int W = a.W, H = a.H, wx = 2 * a.nax + 1;
    const bool count_all = !(a.arith == 0 && uniform_branch);
    int pa = 0, pb = 255, zeros = 0;
    // one reduction step of the fold: the first pending sample (in window order) that lies strictly inside (pa, pb) moves a bound
    auto fold = [&](int vl, int vr, int keyl, int keyr) {
        int done = -1;
        while (true) {
            const bool pl = vl > pa && vl < pb && keyl > done;
            const bool pr = vr > pa && vr < pb && keyr > done;
            const unsigned key = pl ? (unsigned)keyl : (pr ? (unsigned)keyr : 0xFFFFFFFFu);
            const unsigned m = __reduce_min_sync(0xFFFFFFFFu, key);
            if (m == 0xFFFFFFFFu) break;
            const int v = (int)(m & 255u);
            done = (int)m;
            if (v - pa > pb - v) pb = v;
            else if (v - pa < pb - v) pa = v;
        }
    };
    if (wx <= 64) {
        // windows of up to 64 columns (the default 64 x 3): the two 32-column halves' validity does not depend on the row and is
        // worked out once per window; the four samples of a row are fetched together
        const int xa = cx - a.nax + lane, xb = xa + 32;
        const bool ina = lane < wx && xa >= 0 && xa <= W - 1, inb = lane + 32 < wx && xb >= 0 && xb <= W - 1;
        const bool hra = ina && xa - shift >= 0 && xa - shift <= W - 1, hrb = inb && xb - shift >= 0 && xb - shift <= W - 1;
        const bool hla = ina && (!occ || !hra), hlb = inb && (!occ || !hrb);
        const int kla = (2 * lane) << 8, kra = kla + 256, klb = (2 * lane + 64) << 8, krb = klb + 256;
        const uint8_t *pl0 = src.sL + (max(cy - a.nay, 0) - src.oy) * src.RW + (cx - a.nax - src.ox) + lane;
        const uint8_t *pr0 = src.sR + (pl0 - src.sL);
        for (int yy = max(cy - a.nay, 0); yy <= min(cy + a.nay, H - 1); yy++, pl0 += src.RW, pr0 += src.RW) {
            const int vla = hla ? (int)pl0[0] : -1, vra = hra ? (int)pr0[0] : -1;
            const int vlb = hlb ? (int)pl0[32] : -1, vrb = hrb ? (int)pr0[32] : -1;
            zeros += (vla == 0) + (vra == 0) + (vlb == 0) + (vrb == 0);
            fold(vla, vra, kla | (vla & 255), kra | (vra & 255));
            if (wx > 32) fold(vlb, vrb, klb | (vlb & 255), krb | (vrb & 255));
        }
    } else {
        const int keyl0 = (2 * lane) << 8, keyr0 = (2 * lane + 1) << 8;
        for (int yy = max(cy - a.nay, 0); yy <= min(cy + a.nay, H - 1); yy++) {
            const int base = (yy - src.oy) * src.RW + (cx - a.nax - src.ox);
            for (int c0 = 0; c0 < wx; c0 += 32) {
                const int dx = c0 + lane, xx = cx - a.nax + dx, xr = xx - shift;
                const bool in = dx < wx && xx >= 0 && xx <= W - 1;
                const bool has_r = in && xr >= 0 && xr <= W - 1;
                const bool has_l = in && (!occ || !has_r);
                const int vl = has_l ? (int)src.sL[base + dx] : -1;
                const int vr = has_r ? (int)src.sR[base + dx] : -1;
                zeros += (vl == 0) + (vr == 0);
                fold(vl, vr, keyl0 | (vl & 255), keyr0 | (vr & 255));
            }
        }
    }
    if (count_all && __reduce_add_sync(0xFFFFFFFFu, zeros) == 256)
        return max_dist_colour(a, src, cy, cx, shift, occ, uniform_branch, lane);
    return (double)(pa + pb) / 2.0;
}

// ---- maxDistance, wavefront version: one warp per (frame, channel, hint row), rows pipelined behind each other -----
// The scan is sequential, but two hints only interact when one writes what the other reads or writes.  Writes of a hint
// stay within rows y-n..y+n and columns x-n..x+n (left) / x-d1-n..x-d0+n (right), reads within n+nay rows and n+nax
// columns of those, so hints of rows further apart than RD = 2n+nay never interact and a hint of row y only has to wait
// for the LAST hint of each row y-1..y-RD whose footprint overlaps its own (vpp_md_deps_kernel finds them; rows run in
// scan order, so "hint k' of that row is done" covers all earlier ones).  Rows are handed out through a ticket counter in
// raster order, so everything a row waits for is already running or finished: no deadlock.  Every hint is still applied
// after all earlier hints it could observe and before all later hints that could observe it: bit-exact.
// A hint's working set (the union of its patch pixels' windows in both images) is staged once in shared memory; the
// folds of the 9 patch pixels and lane 0's blends then run out of it (blends write through to global memory).
struct MdWs {
    uint16_t *dep;       // [n][H][RD][W] per hint (parallel to hx): 1 + index of the last interacting hint of row y-1-r, 0 = none
    int *prog;           // [n*C][H] hints of that row already applied
    int *ticket;         // [1]
};

static size_t md_ws_layout(int H, int W, int C, int n, int RD, void *base, size_t base_off, MdWs *ws)
{
    size_t off = align256(base_off);
    char *b = (char *)base;
    auto take = [&](size_t bytes) { size_t o = off; off += align256(bytes); return b ? b + o : (char *)nullptr; };
    uint16_t *dep = (uint16_t *)take((size_t)n * H * RD * W * 2);
    int *prog = (int *)take(((size_t)n * C * H + 64) * 4);
    if (ws) { ws->dep = dep; ws->prog = prog; ws->ticket = prog + (size_t)n * C * H; }
    return off;
}

struct MdFoot {                    // column footprints of one hint; intervals are clipped to the image, empty = hi < lo
    int wl_lo, wl_hi, fl_lo, fl_hi;        // left image: written / touched
    int wr_lo, wr_hi, fr_lo, fr_hi;        // right image: written (and read back by the blend) / touched
    int wrap_lo;                           // right-image accesses at negative columns wrap to [wrap_lo, W-1]; W = none
};
__device__ __forceinline__ MdFoot md_foot(const VppArgs &a, int x, float gv)
{
    const HintGeom hg = hint_geom(a, gv, x);
    const int W = a.W, n = a.n, m = a.n + a.nax;
    MdFoot f;
    f.wl_lo = max(x - n, 0); f.wl_hi = min(x + n, W - 1);
    f.fl_lo = max(x - m, 0); f.fl_hi = min(x + m, W - 1);
    const int lo = min(hg.xd1, hg.xd) - n, hi = max(hg.xd0, hg.xd) + n;
    f.wr_lo = max(lo, 0); f.wr_hi = min(hi, W - 1);
    f.fr_lo = max(min(lo, hg.xd - m), 0); f.fr_hi = min(max(hi, hg.xd + m), W - 1);
    f.wrap_lo = (lo < 0 && hi >= 0) ? max(W + lo, 0) : W;
    return f;
}
__device__ __forceinline__ bool md_ov(int alo, int ahi, int blo, int bhi) { return max(alo, blo) <= min(ahi, bhi); }
__device__ __forceinline__ bool md_conflict(const MdFoot &p, const MdFoot &q, int W)
{
    if (md_ov(p.wl_lo, p.wl_hi, q.fl_lo, q.fl_hi) || md_ov(p.fl_lo, p.fl_hi, q.wl_lo, q.wl_hi)) return true;
    if (md_ov(p.wr_lo, p.wr_hi, q.fr_lo, q.fr_hi) || md_ov(p.fr_lo, p.fr_hi, q.wr_lo, q.wr_hi)) return true;
    if (p.wrap_lo < W && (q.wrap_lo < W || q.fr_hi >= p.wrap_lo)) return true;
    if (q.wrap_lo < W && p.fr_hi >= q.wrap_lo) return true;
    return false;
}

// one CTA per (frame, row): for every hint of the row, the last interacting hint of each of the RD rows above
__global__ void __launch_bounds__(128) vpp_md_deps_kernel(const float *__restrict__ g, VppWs ws, MdWs md, VppArgs a, int RD)
{
    const long row = blockIdx.x;
    const int W = a.W, H = a.H;
    const int y = (int)(row % H);
    const int cnt = ws.cnt[row];
    const uint16_t *hx = ws.hx + row * W;
    for (int k = threadIdx.x; k < cnt; k += blockDim.x) {
        const int x = hx[k];
        const MdFoot me = md_foot(a, x, g[row * W + x]);
        for (int r = 0; r < RD; r++) {
            int dep = 0;
            if (y - 1 - r >= 0) {
                const long prow = row - 1 - r;
                const uint16_t *phx = ws.hx + prow * W;
                for (int kk = ws.cnt[prow] - 1; kk >= 0; kk--) {
                    const int px = phx[kk];
                    if (md_conflict(me, md_foot(a, px, g[prow * W + px]), W)) { dep = kk + 1; break; }
                }
            }
            md.dep[(row * RD + r) * W + k] = (uint16_t)dep;
        }
    }
}

__device__ __forceinline__ int md_ld_acquire(const int *p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// Raised by a dependency wait of the maxDistance wavefront that timed out (a protocol error, or the device so oversubscribed
// that the rows ahead made no progress for a minute).  The scan then continues with undefined results instead of trapping the
// context; the host reads the flag with vppb200_async_error().
__device__ unsigned int g_md_abort = 0;

// long dependency wait (the rows far ahead of the wavefront): bounded, so a protocol error cannot hang the device
__device__ __noinline__ void md_long_wait(const int *p, int need)
{
    for (unsigned spins = 0; spins < (1u << 26); spins++) {
        const int got = md_ld_acquire(p);           // every lane polls its own (always valid) word: no divergence in the loop
        if (!__any_sync(0xFFFFFFFFu, got < need)) return;
        if ((spins & 1023u) == 1023u && *(volatile unsigned int *)&g_md_abort != 0u) return;
        __nanosleep(1024u);
    }
    g_md_abort = 1u;
}
__device__ __forceinline__ void md_st_release(int *p, int v)
{
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

static constexpr int MD_IMAX = 11;

struct MdSplat {
    const VppArgs &a;
    uint8_t *lrow, *rrow;      // global row pointers at channel j
    uint8_t *sl, *sr;          // region row of the same image row
    int ox, shift, RW;
    __device__ __forceinline__ uint8_t getL(int x) const { return sl[x - ox]; }                 // patch pixels are inside the region
    __device__ __forceinline__ void setL(int x, uint8_t v) const { sl[x - ox] = v; lrow[(long)x * a.C] = v; }
    __device__ __forceinline__ uint8_t getR(int x) const
    {
        if (x < 0) x += a.W;
        const int c = x + shift - ox;
        return (c >= 0 && c < RW) ? sr[c] : __ldcg(rrow + (long)x * a.C);
    }
    __device__ __forceinline__ void setR(int x, uint8_t v) const
    {
        if (x < 0) x += a.W;
        const int c = x + shift - ox;
        if (c >= 0 && c < RW) sr[c] = v;
        rrow[(long)x * a.C] = v;
    }
};

static constexpr int MD_MINB = 12;      // minimum resident CTAs (one warp each) per SM: caps the wavefront kernel's registers
__global__ void __launch_bounds__(32, MD_MINB) vpp_max_dist_wave_kernel(uint8_t *l, uint8_t *r, const float *__restrict__ g,
                                                               const uint8_t *__restrict__ g_occ, VppWs ws, MdWs md, VppArgs a,
                                                               int units, int RD)
{
    extern __shared__ uint8_t md_smem[];
    const int lane = threadIdx.x;
    const int W = a.W, H = a.H, C = a.C, n = a.n;
    const int RH = 2 * (n + a.nay) + 1, RW = 2 * (n + a.nax) + 1;
    uint8_t *sL = md_smem, *sR = md_smem + RH * RW;
    const long total = (long)units * H;
    int pos[MD_IMAX];                 // region position lane + 32 i as (row << 16 | column); row >= RH = beyond the region
#pragma unroll
    for (int i = 0; i < MD_IMAX; i++) {
        const int p = lane + 32 * i;
        pos[i] = ((p / RW) << 16) | (p % RW);
    }
    while (true) {
        long t = 0;
        if (lane == 0) t = atomicAdd(md.ticket, 1);
        t = __shfl_sync(0xFFFFFFFFu, (int)t, 0);
        if (t >= total) return;
        const int y = (int)(t / units), unit = (int)(t % units);
        const int j = unit % C;
        const long f = unit / C;
        const long row = f * H + y;
        const int cnt = ws.cnt[row];
        if (cnt == 0) continue;
        uint8_t *limg = l + f * (long)H * W * C + j, *rimg = r + f * (long)H * W * C + j;
        int *prog = md.prog + (long)unit * H;
        const uint16_t *hx = ws.hx + row * W;
        // hint k+1's column, value, mask and dependencies are fetched while hint k is folded; lane rr holds the
        // dependency on row y-1-rr and polls it itself
        auto fetch = [&](int k, int &x, float &gv, bool &occ, int &need) {
            x = hx[k];
            gv = g[row * W + x];
            occ = g_occ[row * W + x] != 0;
            need = (lane < RD && y - 1 - lane >= 0) ? (int)md.dep[(row * RD + lane) * W + k] : 0;
        };
        int nx_x, nx_need;
        float nx_gv;
        bool nx_occ;
        fetch(0, nx_x, nx_gv, nx_occ, nx_need);
        const int *mydep = prog + max(y - 1 - lane, 0);
        for (int k = 0; k < cnt; k++) {
            const int x = nx_x, need = nx_need;
            const float gv = nx_gv;
            const bool occ = nx_occ;
            const HintGeom hg = hint_geom(a, gv, x);
            const int shift = x - hg.xd;
            // wait for the hints of the rows above that interact with this one
            {
                unsigned ns = 32;
                while (__any_sync(0xFFFFFFFFu, md_ld_acquire(mydep) < need)) {       // need == 0: no dependency (progress >= 0)
                    if (ns > 1024u) { md_long_wait(mydep, need); break; }      // (kept out of line: the short waits are the hot path)
                    __nanosleep(ns);
                    ns *= 2;
                }
                __syncwarp();                         // ... which orders every lane's loads below
            }
            if (k + 1 < cnt) fetch(k + 1, nx_x, nx_gv, nx_occ, nx_need);
            // stage the working set: all loads first (IMAX x 32 positions cover the default 5 x 67 region), then the stores
            const int oy = y - n - a.nay, ox = x - n - a.nax;
            if (RH * RW <= 32 * MD_IMAX) {
                uint8_t vl[MD_IMAX], vr[MD_IMAX];
#pragma unroll
                for (int i = 0; i < MD_IMAX; i++) {
                    const int ry = pos[i] >> 16, c = pos[i] & 0xFFFF;
                    const int yy = oy + ry, xx = ox + c, xr = xx - shift;
                    const bool yin = ry < RH && yy >= 0 && yy <= H - 1;
                    vl[i] = 0; vr[i] = 0;               // (the right sample is staged even where xx is outside: the blends read it)
                    if (yin && xx >= 0 && xx <= W - 1) vl[i] = __ldcg(limg + ((long)yy * W + xx) * C);
                    if (yin && xr >= 0 && xr <= W - 1) vr[i] = __ldcg(rimg + ((long)yy * W + xr) * C);
                }
#pragma unroll
                for (int i = 0; i < MD_IMAX; i++) {
                    const int ry = pos[i] >> 16, c = pos[i] & 0xFFFF;
                    if (ry < RH) { sL[ry * RW + c] = vl[i]; sR[ry * RW + c] = vr[i]; }
                }
            } else {
                for (int ry = 0; ry < RH; ry++) {
                    const int yy = oy + ry;
                    const bool yin = yy >= 0 && yy <= H - 1;
                    const uint8_t *lp = limg + (long)yy * W * C, *rp = rimg + (long)yy * W * C;
                    for (int c = lane; c < RW; c += 32) {
                        const int xx = ox + c, xr = xx - shift;
                        uint8_t vl = 0, vr = 0;
                        if (yin && xx >= 0 && xx <= W - 1) vl = __ldcg(lp + (long)xx * C);
                        if (yin && xr >= 0 && xr <= W - 1) vr = __ldcg(rp + (long)xr * C);
                        sL[ry * RW + c] = vl; sR[ry * RW + c] = vr;
                    }
                }
            }
            __syncwarp();
            const MdRegionSrc src{sL, sR, oy, ox, RW};
            const int nh = patch_radius(a, f, gv);
            double pv = 0.0;
            if (a.uniform) pv = md_colour_region(a, src, y, x, shift, occ, true, lane);
            for (int yw = -nh; yw <= nh; yw++) {
                if (y + yw < 0 || y + yw > H - 1) continue;
                for (int xw = -nh; xw <= nh; xw++) {
                    if (x + xw < 0 || x + xw > W - 1) continue;
                    if (!patch_keep(a, f, gv, y + yw, x + xw)) continue;
                    if (!a.uniform) pv = md_colour_region(a, src, y + yw, x + xw, shift, occ, false, lane);
                    if (lane == 0) {
                        const int ry = y + yw - oy;
                        MdSplat s{a, limg + ((long)(y + yw) * W) * C, rimg + ((long)(y + yw) * W) * C, sL + ry * RW, sR + ry * RW,
                                  ox, shift, RW};
                        splat_pixel<false>(s, pv, x + xw, hg.xd0 + xw, hg.xd1 + xw, hg.xd + xw, occ, hg.b32, hg.b64);
                    }
                    __syncwarp();                     // lane 0's updates of the region are visible to the next fold
                }
            }
            if (lane == 0) md_st_release(prog + y, k + 1);
        }
    }
}

// gt_reshape (pyx:352-371): raster-order compaction to (x, y, d, 1); reuses the per-row lists (direction = 1)
__global__ void gt_reshape_kernel(const float *__restrict__ gt, VppWs ws, int W, int H, float *__restrict__ out, int32_t *count_out)
{
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= H) return;
    const long long base = ws.hbase[y];
    const int cnt = ws.cnt[y];
    for (int k = 0; k < cnt; k++) {
        const int x = ws.hx[(long)y * W + k];
        float4 v = make_float4((float)x, (float)y, gt[(long)y * W + x], 1.0f);
        reinterpret_cast<float4 *>(out)[base + k] = v;
    }
    if (y == H - 1 && count_out) *count_out = (int32_t)(base + cnt);
}

static int prepare_hints(const float *g, int W, int H, int n_patch, int direction, const VppWs &ws, int32_t *n_hints_out, int n,
                         cudaStream_t st, const VppArgs *adaptive = nullptr)
{
    const long rows = (long)n * H;
    vpp_compact_rows_kernel<<<cdiv(rows * 32, 128), 128, 0, st>>>(g, ws, W, H, n_patch, direction, rows);
    VPP_LAUNCH_CHECK("vpp_compact_rows_kernel");
    if (adaptive) {          // draws per hint = kept in-image patch pixels: recount (hpre, draws) before the row scan
        vpp_adaptive_counts_kernel<<<cdiv(rows * 32, 128), 128, 0, st>>>(g, ws, *adaptive, rows);
        VPP_LAUNCH_CHECK("vpp_adaptive_counts_kernel");
    }
    vpp_scan_rows_kernel<<<cdiv((long)n * 32, 128), 128, 0, st>>>(ws, H, n, n_hints_out);
    VPP_LAUNCH_CHECK("vpp_scan_rows_kernel");
    return VPPB200_OK;
}

static int g_vpp_rows_on = 1;       // test hook: 0 = ordered per-row replay only
void vpp_set_rows_kernel(int on) { g_vpp_rows_on = on != 0; }
static int g_vpp_md_wave = 1;       // test hook: 0 = maxDistance by the serial one-warp-per-(frame, channel) kernel only
int vpp_take_md_abort_flag(int *out)
{
    unsigned int v = 0, zero = 0;
    VPP_CUDA_TRY(cudaMemcpyFromSymbol(&v, g_md_abort, sizeof v));
    if (v) VPP_CUDA_TRY(cudaMemcpyToSymbol(g_md_abort, &zero, sizeof zero));
    *out = v != 0;
    return VPPB200_OK;
}

void vpp_set_md_wave(int on) { g_vpp_md_wave = on > 0; }

static VppArgs make_args(int W, int H, int C, int uniform, int wsize, int wax, int way, int direction, double c, double c_occ,
                         int discard, int interpolate, int arith)
{
    VppArgs a;
    a.W = W; a.H = H; a.C = C; a.uniform = uniform != 0; a.n = (wsize - 1) / 2; a.nax = (wax - 1) / 2; a.nay = (way - 1) / 2;
    a.direction = direction; a.discard = discard != 0; a.interpolate = interpolate != 0; a.arith = arith;
    a.c32 = (float)c; a.cocc32 = (float)c_occ; a.c64 = c; a.cocc64 = c_occ;
    a.filled = nullptr; a.thr = nullptr; a.nthr = 0;
    a.y0 = 0; a.y1 = H;
    return a;
}

}  // namespace vppb200

using namespace vppb200;

extern "C" size_t vppb200_vpp_workspace_bytes(int H, int W, int C, int n)
{
    (void)C;
    if (H <= 0 || W <= 0 || n <= 0) return 0;
    return vpp_ws_layout(H, W, n, nullptr, nullptr);
}

static int scan_rnd_impl(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color, int wsize,
                         int direction, double c, double c_occ, const uint8_t *g_occ, int discard_occluded,
                         int interpolate, int arith, const uint8_t *pattern, const int64_t *pattern_offsets,
                         uint64_t rng_seed, int32_t *n_hints_out, void *workspace, size_t workspace_bytes, int n, void *stream,
                         const float *filled_g, const float *thresholds, int n_thresholds, int row_begin = 0, int row_end = -1)
{
    if (row_end < 0) row_end = H;
    if (!l || !r || !g || !g_occ || (pattern && !pattern_offsets) || W <= 0 || H <= 0 || C <= 0 || n <= 0 || wsize < 1 || W > 65535 ||
        (arith != 0 && arith != 1) || (thresholds && n_thresholds != wsize - 1) || row_begin < 0 || row_end > H || row_begin > row_end)
        return VPPB200_ERR_ARG;
    if (!workspace || workspace_bytes < vpp_ws_layout(H, W, n, nullptr, nullptr)) return VPPB200_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    VppWs ws;
    vpp_ws_layout(H, W, n, workspace, &ws);
    VppArgs a = make_args(W, H, C, uniform_color, wsize, 1, 1, direction, c, c_occ, discard_occluded, interpolate, arith);
    a.y0 = row_begin; a.y1 = row_end;
    if (filled_g || thresholds) {
        // adaptive patches: recounted stream positions, ordered per-row replay with per-hint radius and keep test
        a.filled = filled_g; a.thr = thresholds; a.nthr = thresholds ? n_thresholds : 0;
        int rc = prepare_hints(g, W, H, a.n, direction, ws, n_hints_out, n, st, &a);
        if (rc) return rc;
        const long total = (long)n * H * C;
        vpp_rnd_adaptive_kernel<<<cdiv(total, 128), 128, 0, st>>>(l, r, g, g_occ, pattern, pattern_offsets, rng_seed, ws, a, total);
        VPP_LAUNCH_CHECK("vpp_rnd_adaptive_kernel");
        return VPPB200_OK;
    }
    int rc = prepare_hints(g, W, H, a.n, direction, ws, n_hints_out, n, st);
    if (rc) return rc;
    // per-pixel replay for every row it can take; the rows it flags go to the ordered per-row replay
    const RowsCfg cfg{4096, 1024};
    const size_t smem = vr_smem_bytes(W, cfg);
    int dev = 0, smem_optin = 0;
    VPP_CUDA_TRY(cudaGetDevice(&dev));
    VPP_CUDA_TRY(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    // (the per-pixel replay addresses a frame's pattern stream with 32 bits)
    const bool rows_kernel = g_vpp_rows_on && smem <= (size_t)smem_optin && (long)n * H < (1L << 31) &&
                             (double)C * W * H * wsize * wsize < 4.0e9;
    if (rows_kernel) {
        VPP_CUDA_TRY(cudaFuncSetAttribute(vpp_rnd_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        vpp_rnd_rows_kernel<<<(unsigned)((long)n * H), VR_NT, smem, st>>>(l, r, g, g_occ, pattern, pattern_offsets, rng_seed, ws, a, cfg);
        VPP_LAUNCH_CHECK("vpp_rnd_rows_kernel");
    }
    const long total = (long)n * H * C;
    vpp_rnd_replay_kernel<<<cdiv(total, 128), 128, 0, st>>>(l, r, g, g_occ, pattern, pattern_offsets, rng_seed, ws, a, total,
                                                            rows_kernel ? 1 : 0);
    VPP_LAUNCH_CHECK("vpp_rnd_replay_kernel");
    return VPPB200_OK;
}

extern "C" int vppb200_vpp_scan_rnd(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color, int wsize,
                                    int direction, double c, double c_occ, const uint8_t *g_occ, int discard_occluded,
                                    int interpolate, int arith, const uint8_t *pattern, const int64_t *pattern_offsets,
                                    uint64_t rng_seed, int32_t *n_hints_out, void *workspace, size_t workspace_bytes, int n, void *stream)
{
    return scan_rnd_impl(l, r, g, W, H, C, uniform_color, wsize, direction, c, c_occ, g_occ, discard_occluded, interpolate, arith,
                         pattern, pattern_offsets, rng_seed, n_hints_out, workspace, workspace_bytes, n, stream, nullptr, nullptr, 0);
}

extern "C" int vppb200_vpp_scan_rnd_adaptive(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color, int wsize,
                                             int direction, double c, double c_occ, const uint8_t *g_occ, int discard_occluded,
                                             int interpolate, int arith, const uint8_t *pattern, const int64_t *pattern_offsets,
                                             uint64_t rng_seed, const float *filled_g, const float *patch_thresholds,
                                             int n_thresholds, int32_t *n_hints_out, void *workspace, size_t workspace_bytes, int n,
                                             void *stream)
{
    return scan_rnd_impl(l, r, g, W, H, C, uniform_color, wsize, direction, c, c_occ, g_occ, discard_occluded, interpolate, arith,
                         pattern, pattern_offsets, rng_seed, n_hints_out, workspace, workspace_bytes, n, stream, filled_g,
                         patch_thresholds, n_thresholds);
}

extern "C" int vppb200_vpp_scan_rnd_rows(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color, int wsize,
                                         int direction, double c, double c_occ, const uint8_t *g_occ, int discard_occluded,
                                         int interpolate, int arith, const uint8_t *pattern, const int64_t *pattern_offsets,
                                         uint64_t rng_seed, int row_begin, int row_end, int32_t *n_hints_out, void *workspace,
                                         size_t workspace_bytes, int n, void *stream)
{
    return scan_rnd_impl(l, r, g, W, H, C, uniform_color, wsize, direction, c, c_occ, g_occ, discard_occluded, interpolate, arith,
                         pattern, pattern_offsets, rng_seed, n_hints_out, workspace, workspace_bytes, n, stream, nullptr, nullptr, 0,
                         row_begin, row_end);
}

extern "C" int vppb200_bilateral_filling(const float *dmap, const uint8_t *gray, float *out, int W, int H, int n_patch,
                                         const double *weights, double th, int n, void *stream)
{
    if (!dmap || !gray || !out || !weights || W <= 0 || H <= 0 || n_patch < 0 || n <= 0) return VPPB200_ERR_ARG;
    const long total = (long)n * H * W;
    bilateral_filling_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(dmap, gray, out, W, H, n_patch, weights, th, total);
    VPP_LAUNCH_CHECK("bilateral_filling_kernel");
    return VPPB200_OK;
}

extern "C" int vppb200_bgr2gray(const uint8_t *src, uint8_t *gray, int W, int H, int C, int n, void *stream)
{
    if (!src || !gray || W <= 0 || H <= 0 || C <= 0 || n <= 0) return VPPB200_ERR_ARG;
    const long total = (long)n * H * W;
    bgr2gray_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(src, gray, C, total);
    VPP_LAUNCH_CHECK("bgr2gray_kernel");
    return VPPB200_OK;
}

extern "C" int vppb200_distance_patch_thresholds(const float *g, int W, int H, const float *ratio_steps, int wsize,
                                                 float *patch_thresholds, int32_t *status, int n, void *stream)
{
    if (!g || W <= 0 || H <= 0 || wsize < 1 || n <= 0 || (wsize > 1 && (!ratio_steps || !patch_thresholds)))
        return VPPB200_ERR_ARG;
    distance_patch_thresholds_kernel<<<n, 1024, 0, (cudaStream_t)stream>>>(g, (long)W * H, ratio_steps, wsize - 1,
                                                                           patch_thresholds, status);
    VPP_LAUNCH_CHECK("distance_patch_thresholds_kernel");
    return VPPB200_OK;
}

static int scan_max_dist_impl(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color, int wsize,
                              int wsize_agg_x, int wsize_agg_y, int direction, double c, double c_occ,
                              const uint8_t *g_occ, int discard_occluded, int interpolate, int arith,
                              int32_t *n_hints_out, void *workspace, size_t workspace_bytes, int n, void *stream,
                              const float *filled_g, const float *thresholds, int n_thresholds)
{
    if (!l || !r || !g || !g_occ || W <= 0 || H <= 0 || C <= 0 || n <= 0 || wsize < 1 || wsize_agg_x < 1 || wsize_agg_y < 1 ||
        W > 65535 || (arith != 0 && arith != 1) || (thresholds && n_thresholds != wsize - 1))
        return VPPB200_ERR_ARG;
    if (!workspace || workspace_bytes < vpp_ws_layout(H, W, n, nullptr, nullptr)) return VPPB200_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    VppWs ws;
    vpp_ws_layout(H, W, n, workspace, &ws);
    VppArgs a = make_args(W, H, C, uniform_color, wsize, wsize_agg_x, wsize_agg_y, direction, c, c_occ, discard_occluded,
                          interpolate, arith);
    a.filled = filled_g; a.thr = thresholds; a.nthr = thresholds ? n_thresholds : 0;     // footprints stay those of the full patch
    int rc = prepare_hints(g, W, H, a.n, direction, ws, n_hints_out, n, st);
    if (rc) return rc;
    const int total = n * C;
    // wavefront kernel when the caller's workspace holds the dependency table (vppb200_vpp_max_dist_workspace_bytes) and a
    // hint's working set fits shared memory; the serial one-warp-per-(frame, channel) kernel otherwise
    const int RD = 2 * a.n + a.nay;
    const size_t base_bytes = vpp_ws_layout(H, W, n, nullptr, nullptr);
    const size_t smem = 2 * (size_t)(2 * (a.n + a.nay) + 1) * (2 * (a.n + a.nax) + 1);
    int dev = 0, smem_optin = 0, sms = 0;
    VPP_CUDA_TRY(cudaGetDevice(&dev));
    VPP_CUDA_TRY(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    VPP_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const bool wave = g_vpp_md_wave && RD >= 1 && RD <= 32 && smem <= (size_t)smem_optin && (long)total * H < (1L << 30) &&
                      workspace_bytes >= md_ws_layout(H, W, C, n, RD, nullptr, base_bytes, nullptr);
    if (wave) {
        MdWs md;
        md_ws_layout(H, W, C, n, RD, workspace, base_bytes, &md);
        VPP_CUDA_TRY(cudaMemsetAsync(md.prog, 0, ((size_t)total * H + 64) * 4, st));
        vpp_md_deps_kernel<<<(unsigned)((long)n * H), 128, 0, st>>>(g, ws, md, a, RD);
        VPP_LAUNCH_CHECK("vpp_md_deps_kernel");
        VPP_CUDA_TRY(cudaFuncSetAttribute(vpp_max_dist_wave_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const long rows = (long)total * H;
        const long resident = (long)sms * (smem <= 4096 ? 32 : max((size_t)1, (size_t)200 * 1024 / (smem + 1024)));
        vpp_max_dist_wave_kernel<<<(unsigned)min(rows, resident), 32, smem, st>>>(l, r, g, g_occ, ws, md, a, total, RD);
        VPP_LAUNCH_CHECK("vpp_max_dist_wave_kernel");
        return VPPB200_OK;
    }
    vpp_max_dist_kernel<<<total, 32, 0, st>>>(l, r, g, g_occ, ws, a, total);
    VPP_LAUNCH_CHECK("vpp_max_dist_kernel");
    return VPPB200_OK;
}

extern "C" int vppb200_vpp_scan_max_dist(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color, int wsize,
                                         int wsize_agg_x, int wsize_agg_y, int direction, double c, double c_occ,
                                         const uint8_t *g_occ, int discard_occluded, int interpolate, int arith,
                                         int32_t *n_hints_out, void *workspace, size_t workspace_bytes, int n, void *stream)
{
    return scan_max_dist_impl(l, r, g, W, H, C, uniform_color, wsize, wsize_agg_x, wsize_agg_y, direction, c, c_occ, g_occ,
                              discard_occluded, interpolate, arith, n_hints_out, workspace, workspace_bytes, n, stream, nullptr,
                              nullptr, 0);
}

extern "C" int vppb200_vpp_scan_max_dist_adaptive(uint8_t *l, uint8_t *r, const float *g, int W, int H, int C, int uniform_color,
                                                  int wsize, int wsize_agg_x, int wsize_agg_y, int direction, double c, double c_occ,
                                                  const uint8_t *g_occ, int discard_occluded, int interpolate, int arith,
                                                  const float *filled_g, const float *patch_thresholds, int n_thresholds,
                                                  int32_t *n_hints_out, void *workspace, size_t workspace_bytes, int n, void *stream)
{
    return scan_max_dist_impl(l, r, g, W, H, C, uniform_color, wsize, wsize_agg_x, wsize_agg_y, direction, c, c_occ, g_occ,
                              discard_occluded, interpolate, arith, n_hints_out, workspace, workspace_bytes, n, stream, filled_g,
                              patch_thresholds, n_thresholds);
}

extern "C" size_t vppb200_vpp_max_dist_workspace_bytes(int H, int W, int C, int wsize, int wsize_agg_y, int n)
{
    if (H <= 0 || W <= 0 || C <= 0 || n <= 0 || wsize < 1 || wsize_agg_y < 1) return 0;
    const int RD = 2 * ((wsize - 1) / 2) + (wsize_agg_y - 1) / 2;
    const size_t base = vpp_ws_layout(H, W, n, nullptr, nullptr);
    return RD >= 1 ? md_ws_layout(H, W, C, n, RD, nullptr, base, nullptr) : base;
}

extern "C" int vppb200_gt_reshape(const float *gt, int W, int H, float *out, int32_t *count_out, void *workspace,
                                  size_t workspace_bytes, void *stream)
{
    if (!gt || !out || W <= 0 || H <= 0 || W > 65535) return VPPB200_ERR_ARG;
    if (!workspace || workspace_bytes < vpp_ws_layout(H, W, 1, nullptr, nullptr)) return VPPB200_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    VppWs ws;
    vpp_ws_layout(H, W, 1, workspace, &ws);
    int rc = prepare_hints(gt, W, H, 0, 1, ws, nullptr, 1, st);
    if (rc) return rc;
    gt_reshape_kernel<<<cdiv(H, 128), 128, 0, st>>>(gt, ws, W, H, out, count_out);
    VPP_LAUNCH_CHECK("gt_reshape_kernel");
    return VPPB200_OK;
}
