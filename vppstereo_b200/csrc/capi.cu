// capi.cu -- extern "C" entry points of include/vppstereo_b200.h: argument validation (mirroring the TypeError classes of
// the reference wrapper RSGM/pyrSGM.cpp), workspace carving and the compute_rsgm stage pipeline
// (models/rsgm/rsgm.py:250-294).  The VPP entry points live in vpp.cu.
#include "common.cuh"

#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>
#include <xmmintrin.h>

namespace vppb200 {

static std::atomic<uint64_t> g_launches{0};
static thread_local char g_err[256] = "";

void note_launch(int k) { g_launches.fetch_add((uint64_t)k, std::memory_order_relaxed); }

int cuda_fail(const char *what, cudaError_t e)
{
    snprintf(g_err, sizeof g_err, "%s: %s", what, cudaGetErrorString(e));
    return VPPB200_ERR_CUDA;
}

// rcp_nz_ss(-2k) (RSGM/StereoBMHelper.cpp:752-756): RCPSS is a vendor-specific table instruction, so the reference's sub-pixel
// disparities depend on the CPU it runs on.  Default here: the fixed table of Intel's approximation (a function of the
// operand's exponent and top 11 mantissa bits, tools/make_rcp_table.py), so that every host and every rank of a sharded run
// produce the same numbers.  VPPB200_TUNE_RCP_HOST = 1 selects the RCPSS of the host CPU instead (parity tests against a
// reference compiled on that host).
static const uint32_t kRcpIntelMant[2048] = {
#include "rcp_intel_table.inc"
};
static void fill_rcp_lut_host(float *lut)
{
    lut[0] = 0.0f;
    for (int k = 1; k < 65536; k++) lut[k] = _mm_cvtss_f32(_mm_rcp_ss(_mm_set_ss(2.0f * (float)(-k))));
}
static void fill_rcp_lut_fixed(float *lut)
{
    lut[0] = 0.0f;
    for (int k = 1; k < 65536; k++) {
        const float x = 2.0f * (float)(-k);
        uint32_t b;
        memcpy(&b, &x, 4);
        const uint32_t r = 0x80000000u | ((253u - ((b >> 23) & 0xFFu)) << 23) | kRcpIntelMant[(b >> 12) & 0x7FFu];
        memcpy(&lut[k], &r, 4);
    }
}
static std::atomic<int> g_rcp_host{0};
static void fill_rcp_lut(float *lut) { g_rcp_host.load() ? fill_rcp_lut_host(lut) : fill_rcp_lut_fixed(lut); }

static std::mutex g_lut_mutex;
static float *g_dev_lut[2][64] = {{nullptr}, {nullptr}};   // [fixed | host][device]

const float *device_rcp_lut(cudaStream_t st)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lock(g_lut_mutex);
    const int which = g_rcp_host.load() ? 1 : 0;
    if (!g_dev_lut[which][dev]) {
        static float host[65536];
        which ? fill_rcp_lut_host(host) : fill_rcp_lut_fixed(host);
        float *d = nullptr;
        if (cudaMalloc(&d, sizeof host) != cudaSuccess) return nullptr;
        // synchronous one-time upload: the host table is static and the copy must be complete before first use
        if (cudaMemcpy(d, host, sizeof host, cudaMemcpyHostToDevice) != cudaSuccess) { cudaFree(d); return nullptr; }
        g_dev_lut[which][dev] = d;
    }
    (void)st;
    return g_dev_lut[which][dev];
}

// ---- optional per-stage timing of compute_rsgm (bench.py's live roofline measurement) ----------------------------
struct StageTimer {
    bool enabled = false;
    std::vector<cudaEvent_t> pending;      // groups of N_STAGES+1 events, one group per timed call
    double acc[VPPB200_N_STAGES] = {0};
    int calls = 0;
};
static StageTimer g_timer;
static std::mutex g_timer_mutex;

struct StageMarks {
    cudaEvent_t ev[VPPB200_N_STAGES + 1];
    bool on = false;
    cudaStream_t st;
    int next = 0;
    void begin(cudaStream_t s)
    {
        std::lock_guard<std::mutex> lock(g_timer_mutex);
        on = g_timer.enabled;
        st = s;
        if (!on) return;
        for (auto &e : ev) cudaEventCreate(&e);
        cudaEventRecord(ev[next++], st);
    }
    // stage `stage` ends here; stages that were skipped since the last mark get (almost) zero time
    void done(int stage)
    {
        if (!on) return;
        while (next <= stage + 1 && next <= VPPB200_N_STAGES) cudaEventRecord(ev[next++], st);
    }
    void end()
    {
        if (!on) return;
        done(VPPB200_N_STAGES - 1);
        std::lock_guard<std::mutex> lock(g_timer_mutex);
        for (auto &e : ev) g_timer.pending.push_back(e);
    }
    static void hook(void *ctx, int stage) { static_cast<StageMarks *>(ctx)->done(stage); }
};

// ---- a side stream per device: the left and the right image branches of compute_rsgm (pad/gray/census before the
// cost volume, median/interpolation after WTA) are independent and individually too small to fill the GPU, so the right
// branch is forked onto the side stream and joined back with events (works under stream capture as well).
static std::mutex g_side_mutex;
static cudaStream_t g_side[2][64] = {{nullptr}, {nullptr}};
// which: 0 = front phase (pad/gray/census of the right image), 1 = tail phase (median/interpolation of the right map);
// two streams so that the front of batch k+1 and the tail of batch k do not serialise when they run concurrently
static cudaStream_t side_stream(int which)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lock(g_side_mutex);
    if (!g_side[which][dev] && cudaStreamCreateWithFlags(&g_side[which][dev], cudaStreamNonBlocking) != cudaSuccess) {
        cudaGetLastError();
        g_side[which][dev] = nullptr;
    }
    return g_side[which][dev];
}
// make `to` wait for everything queued on `from` so far
static int stream_chain(cudaStream_t from, cudaStream_t to)
{
    cudaEvent_t e;
    VPP_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    cudaError_t r = cudaEventRecord(e, from);
    if (r == cudaSuccess) r = cudaStreamWaitEvent(to, e, 0);
    cudaEventDestroy(e);                                  // released once the event has completed
    if (r != cudaSuccess) return cuda_fail("stream_chain", r);
    return VPPB200_OK;
}

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// vppb200_sgm_params -> SgmParams; NULL = the reference's effective values.  Host only: runs before any CUDA call.
static int sgm_params_from(const vppb200_sgm_params *q, SgmParams *out)
{
    if (!q) { *out = default_sgm_params(); return VPPB200_OK; }
    auto u16 = [](int v) { return v >= 0 && v <= 65535; };
    if (!u16(q->p1) || !u16(q->p2min) || !u16(q->gamma)) return VPPB200_ERR_ARG;
    if (!std::isfinite(q->alpha) || !(q->alpha >= 0.0f)) return VPPB200_ERR_ARG;     // then P2 in [P2min, max(P2min, gamma)]
    *out = SgmParams{q->p1, q->p2min, q->gamma, q->alpha};
    return VPPB200_OK;
}

struct RsgmWs {
    uint8_t *gray_l, *gray_r, *guide;
    uint32_t *census_l, *census_r;
    uint8_t *dsi;
    uint16_t *S, *S_xyd;
    void *halo;
    float *dl, *dlf, *dr, *drf;
    uint16_t *cost, *rival;                                   // the match info's padded maps (info layout only)
    TailBufs tail;
};

// `sets` buffer sets of everything that crosses a phase boundary (front -> main: guide, cost volume; main -> tail: raw
// left/right disparities), so that the phases of neighbouring batches can run concurrently on different streams; `set`
// selects the one this call uses.  Everything else is private to one phase and exists once.  info: every set also holds the
// padded cost / rival maps of the match info (main -> tail, like dl / dr); without it the layout is the one it always was.
static size_t rsgm_ws_layout(const RsgmDims &d, int n, int sets, int set, void *base, RsgmWs *ws, bool info = false)
{
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) { size_t o = off; off += align256(bytes); return b ? b + o : (char *)nullptr; };
    const size_t np = (size_t)n * d.Hp * d.Wp, nc = (size_t)n * d.H * tail_stride(d.W);
    RsgmWs w;
    w.gray_l = (uint8_t *)take(np); w.gray_r = (uint8_t *)take(np);
    const size_t tv = tile_volume_elems(d.Wp, d.Hp, d.D, n);  // layout T pads the width to 32-column groups
    const size_t vol = tv > np * d.D ? tv : np * d.D;
    w.guide = nullptr; w.dsi = nullptr; w.dl = nullptr; w.dr = nullptr; w.census_l = nullptr; w.census_r = nullptr;
    w.cost = nullptr; w.rival = nullptr;
    for (int k = 0; k < sets; k++) {
        uint8_t *guide = (uint8_t *)take(np), *dsi = (uint8_t *)take(vol);
        float *dl = (float *)take(np * 4), *dr = (float *)take(np * 4);
        // (the census images cross the front -> main boundary too: the forward sweep turns them into the cost volume)
        uint32_t *cl = (uint32_t *)take(np * 4), *cr = (uint32_t *)take(np * 4);
        uint16_t *cost = info ? (uint16_t *)take(np * 2) : nullptr, *rival = info ? (uint16_t *)take(np * 2) : nullptr;
        if (k == set) { w.guide = guide; w.dsi = dsi; w.dl = dl; w.dr = dr; w.census_l = cl; w.census_r = cr; w.cost = cost; w.rival = rival; }
    }
    w.S = (uint16_t *)take(vol * 2);                          // the uint16 S (layout T)
    w.S_xyd = (uint16_t *)take(np * d.D * 2);                 // the reference's xyd order (WTA input, test tap)
    w.halo = (void *)take(sweep_halo_bytes(d.Wp, d.Hp, d.D, n));
    w.dlf = (float *)take(np * 4); w.drf = (float *)take(np * 4);
    w.tail.u8 = (uint8_t *)take(nc); w.tail.label = (int *)take(nc * 4); w.tail.count = (int *)take(nc * 4);
    if (ws) *ws = w;
    return off;
}

}  // namespace vppb200

using namespace vppb200;

extern "C" const char *vppb200_version(void) { return "vppstereo_b200 0.1.0 (sm_100a)"; }
extern "C" const char *vppb200_last_cuda_error(void) { return g_err; }
extern "C" uint64_t vppb200_launch_count(void) { return g_launches.load(); }

extern "C" int vppb200_rcp_lut_host(float *lut_host)
{
    if (!lut_host) return VPPB200_ERR_ARG;
    fill_rcp_lut(lut_host);
    return VPPB200_OK;
}

// glibc TYPE_3 random(): r[i] = r[i-3] + r[i-31] (mod 2^32), output r[i] >> 1.  state34 = the 31-word ring + cursor.
extern "C" int vppb200_glibc_srand(uint32_t *st, uint32_t seed)
{
    if (!st) return VPPB200_ERR_ARG;
    int32_t r[34];
    r[0] = seed == 0 ? 1 : (int32_t)seed;
    for (int i = 1; i < 31; i++) {
        const int64_t hi = r[i - 1] / 127773, lo = r[i - 1] % 127773;
        int64_t word = 16807 * lo - 2836 * hi;
        if (word < 0) word += 2147483647;
        r[i] = (int32_t)word;
    }
    uint32_t ring[31];
    for (int i = 0; i < 31; i++) ring[i] = (uint32_t)r[i];
    // ring is indexed modulo 31; position k holds r[k], next output index is 31 (i.e. slot 0), f = i-3, r = i-31
    for (int i = 0; i < 31; i++) st[i] = ring[i];
    st[31] = 0;    // cursor: slot of r[i-31] == slot to overwrite with r[i]
    st[32] = st[33] = 0;
    uint8_t sink[310];
    // srandom discards 310 outputs; the first 3 steps of the textbook description (r[31..33] = r[i-31]) are the same
    // additive step because glibc starts with fptr = &r[3], rptr = &r[0]:  r[3] += r[0] ...
    // -> use the generic step from the start with the glibc pointer layout.
    st[31] = 0;
    return vppb200_glibc_rand_fill(st, sink, -310);
}

extern "C" int vppb200_glibc_rand_fill(uint32_t *st, uint8_t *out, int64_t n)
{
    if (!st) return VPPB200_ERR_ARG;
    const bool discard = n < 0;
    if (discard) n = -n;
    if (!discard && !out && n > 0) return VPPB200_ERR_ARG;
    uint32_t cur = st[31];            // rptr slot; fptr slot = (cur + 3) % 31
    for (int64_t k = 0; k < n; k++) {
        const uint32_t f = (cur + 3) % 31;
        st[f] += st[cur];
        const uint32_t result = st[f] >> 1;
        if (!discard) out[k] = (uint8_t)(result % 256u);
        cur = (cur + 1) % 31;
    }
    st[31] = cur;
    return VPPB200_OK;
}

extern "C" int vppb200_stage_timing(int enable)
{
    std::lock_guard<std::mutex> lock(g_timer_mutex);
    for (auto &e : g_timer.pending) cudaEventDestroy(e);
    g_timer.pending.clear();
    for (auto &a : g_timer.acc) a = 0;
    g_timer.calls = 0;
    g_timer.enabled = enable != 0;
    return VPPB200_OK;
}

extern "C" int vppb200_stage_times(float *ms_out, int *calls_out)
{
    if (!ms_out) return VPPB200_ERR_ARG;
    std::lock_guard<std::mutex> lock(g_timer_mutex);
    const size_t group = VPPB200_N_STAGES + 1;
    for (size_t g = 0; g + group <= g_timer.pending.size(); g += group) {
        VPP_CUDA_TRY(cudaEventSynchronize(g_timer.pending[g + group - 1]));
        for (int s = 0; s < VPPB200_N_STAGES; s++) {
            float ms = 0;
            VPP_CUDA_TRY(cudaEventElapsedTime(&ms, g_timer.pending[g + s], g_timer.pending[g + s + 1]));
            g_timer.acc[s] += ms;
        }
        g_timer.calls++;
    }
    for (auto &e : g_timer.pending) cudaEventDestroy(e);
    g_timer.pending.clear();
    for (int s = 0; s < VPPB200_N_STAGES; s++) ms_out[s] = (float)g_timer.acc[s];
    if (calls_out) *calls_out = g_timer.calls;
    return VPPB200_OK;
}

extern "C" int vppb200_async_error(void)
{
    int hit = 0, hit_md = 0;
    int rc = sweep_take_abort_flag(&hit);
    if (rc) return rc;
    if ((rc = vpp_take_md_abort_flag(&hit_md))) return rc;
    if (hit_md) {
        snprintf(g_err, sizeof g_err, "vpp_max_dist_wave_kernel: a dependency wait of the row wavefront timed out (results of the affected "
                                      "calls are undefined)");
        return VPPB200_ERR_CUDA;
    }
    if (hit) {
        snprintf(g_err, sizeof g_err, "sgm_v2_kernel: a hand-off wait between the CTAs of a team timed out (results of the affected "
                                      "calls are undefined); were all CTAs of the cooperative grid resident?");
        return VPPB200_ERR_CUDA;
    }
    return VPPB200_OK;
}

extern "C" int vppb200_set_tuning(int key, int value)
{
    switch (key) {
        case VPPB200_TUNE_SGM_MAX_STRIP: sweep_set_max_strip(value); return VPPB200_OK;
        case VPPB200_TUNE_SGM_SWEEP: sweep_set_enabled(value); return VPPB200_OK;
        case VPPB200_TUNE_SGM_CLUSTERS: sweep_set_clusters(value); return VPPB200_OK;
        case VPPB200_TUNE_VPP_ROWS: vpp_set_rows_kernel(value); return VPPB200_OK;
        case VPPB200_TUNE_VPP_MD_WAVE: vpp_set_md_wave(value); return VPPB200_OK;
        case VPPB200_TUNE_SGM_BYTE_SUMS:                         // retired options (the header says why): accepted, no effect
        case VPPB200_TUNE_SGM_FUSE_COST:
        case VPPB200_TUNE_SGM_V_RED:
        case VPPB200_TUNE_SGM_V_SPLIT:
        case VPPB200_TUNE_CENSUS_FUSED: return VPPB200_OK;
        case VPPB200_TUNE_RCP_HOST: g_rcp_host.store(value != 0); return VPPB200_OK;
        default: return VPPB200_ERR_ARG;
    }
}

static int check_wd(int W, int H, int D, int n)
{
    if (W <= 0 || H <= 0 || n <= 0) return VPPB200_ERR_ARG;
    if (W % 16 != 0) return VPPB200_ERR_WIDTH;
    if (D >= 0 && (D <= 0 || D % 8 != 0 || D > 256)) return VPPB200_ERR_DISP;
    return VPPB200_OK;
}

extern "C" int vppb200_census5x5(const uint8_t *src, uint32_t *dst, int W, int H, int n, void *stream)
{
    int rc = check_wd(W, H, -1, n);
    if (rc) return rc;
    if (!src || !dst) return VPPB200_ERR_ARG;
    return launch_census(src, dst, W, H, n, (cudaStream_t)stream);
}

extern "C" int vppb200_cost_census5x5_xyd(const uint32_t *cl, const uint32_t *cr, uint16_t *dsi, int W, int H, int D,
                                          int num_threads, int n, void *stream)
{
    int rc = check_wd(W, H, D, n);
    if (rc) return rc;
    if (num_threads != 1 && num_threads != 2 && num_threads != 4) return VPPB200_ERR_THREADS;
    if (!cl || !cr || !dsi) return VPPB200_ERR_ARG;
    return launch_cost_u16(cl, cr, dsi, W, H, D, n, (cudaStream_t)stream);
}

extern "C" int vppb200_aggregate(const uint8_t *img, const uint16_t *dsi, uint16_t *dsi_agg, int W, int H, int D, int P1,
                                 int P2min, float alpha, int gamma, int honor_params, int n, void *stream)
{
    int rc = check_wd(W, H, D, n);
    if (rc) return rc;
    if (!img || !dsi || !dsi_agg || H < 3) return VPPB200_ERR_ARG;
    const SgmParams prm = honor_params ? SgmParams{P1, P2min, gamma, alpha} : default_sgm_params();   // RSGM/pyrSGM.cpp:519 vs :557-560
    return launch_aggregate_generic(img, dsi, dsi_agg, W, H, D, prm, n, (cudaStream_t)stream);
}

static int check_uniq(float u) { return (u > 1.0f || u <= 0.0f) ? VPPB200_ERR_UNIQUENESS : VPPB200_OK; }

// the uniqueness factor of the _uniq entry points: u finite, 0 < u <= 1 (NaN fails both comparisons); host only
static int uniq_factor(float u, uint32_t *uf)
{
    if (!(u > 0.0f && u <= 1.0f)) return VPPB200_ERR_UNIQUENESS;
    *uf = (uint32_t)(1024.0f * u);
    return VPPB200_OK;
}

extern "C" int vppb200_match_wta(const uint16_t *S, float *disp, int W, int H, int D, float uniqueness, int n, void *stream)
{
    int rc = check_wd(W, H, D, n);
    if (rc) return rc;
    if ((rc = check_uniq(uniqueness))) return rc;
    if (!S || !disp) return VPPB200_ERR_ARG;
    return launch_wta_left(S, disp, W, H, D, n, UNIQ_OFF, (cudaStream_t)stream);
}

extern "C" int vppb200_match_wta_right(const uint16_t *S, float *disp, int W, int H, int D, float uniqueness, int n, void *stream)
{
    int rc = check_wd(W, H, D, n);
    if (rc) return rc;
    if ((rc = check_uniq(uniqueness))) return rc;
    if (!S || !disp) return VPPB200_ERR_ARG;
    return launch_wta_right(S, disp, W, H, D, n, UNIQ_OFF, (cudaStream_t)stream);
}

extern "C" int vppb200_match_wta_uniq(const uint16_t *S, float *disp, int W, int H, int D, float uniqueness, int n, void *stream)
{
    uint32_t uf;
    int rc = check_wd(W, H, D, n);
    if (rc) return rc;
    if ((rc = uniq_factor(uniqueness, &uf))) return rc;
    if (!S || !disp) return VPPB200_ERR_ARG;
    return launch_wta_left(S, disp, W, H, D, n, uf, (cudaStream_t)stream);
}

extern "C" int vppb200_match_wta_right_uniq(const uint16_t *S, float *disp, int W, int H, int D, float uniqueness, int n,
                                            void *stream)
{
    uint32_t uf;
    int rc = check_wd(W, H, D, n);
    if (rc) return rc;
    if ((rc = uniq_factor(uniqueness, &uf))) return rc;
    if (!S || !disp) return VPPB200_ERR_ARG;
    return launch_wta_right(S, disp, W, H, D, n, uf, (cudaStream_t)stream);
}

extern "C" int vppb200_subpixel_refine(const uint16_t *dsi, float *disp, int W, int H, int D, int method, const float *rcp_lut,
                                       int n, void *stream)
{
    int rc = check_wd(W, H, D, n);
    if (rc) return rc;
    if (method != 0 && method != 1) return VPPB200_ERR_METHOD;
    if (!dsi || !disp) return VPPB200_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (!rcp_lut) rcp_lut = device_rcp_lut(st);
    if (!rcp_lut) return cuda_fail("device_rcp_lut", cudaGetLastError());
    return launch_subpixel(dsi, disp, W, H, D, method, rcp_lut, n, st);
}

extern "C" int vppb200_median3x3(const float *src, float *dst, int W, int H, int n, void *stream)
{
    int rc = check_wd(W, H, -1, n);
    if (rc) return rc;
    if (!src || !dst) return VPPB200_ERR_ARG;
    return launch_median(src, dst, W, H, n, (cudaStream_t)stream);
}

extern "C" size_t vppb200_rsgm_workspace_bytes(int H, int W, int C, int D, int n)
{
    if (H <= 0 || W <= 0 || n <= 0 || D <= 0 || D % 8 || D > 256 || (C != 1 && C != 3)) return 0;
    return rsgm_ws_layout(make_dims(H, W, C, D), n, 1, 0, nullptr, nullptr);
}

extern "C" size_t vppb200_rsgm_workspace_bytes_sets(int H, int W, int C, int D, int n, int sets)
{
    if (H <= 0 || W <= 0 || n <= 0 || D <= 0 || D % 8 || D > 256 || (C != 1 && C != 3) || sets < 1 || sets > 4) return 0;
    return rsgm_ws_layout(make_dims(H, W, C, D), n, sets, 0, nullptr, nullptr);
}

// The pipeline in three phases (bit mask `phases`): FRONT = pad/gray/census/cost volume (reads the images, writes the guide
// and the cost volume of buffer set `set`), MAIN = 8-path aggregation + WTA (reads them, writes the raw disparities of the
// set), TAIL = median/interpolation/LR check/speckles/fills (reads those, writes disp_out).  One call may run any subset
// on `stream`; a caller that runs the phases of neighbouring batches on different streams orders them with events
// (vppstereo_b200/pipeline.py).  workspace must have been sized for `sets` sets.  uf: uniqueness factor of MAIN's WTA
// (UNIQ_OFF = none).  state_out != NULL: the match info (all three outputs set, workspace in the info layout), produced by the
// info instantiations of the fused sweep / WTA and of the left-view tail kernels; NULL: exactly the kernels of the plain pipeline.
static int rsgm_phases(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp, const float *hints,
                       const float *validhints, float *disp_out, int H, int W, int C, int D, int flags, const float *rcp_lut,
                       void *workspace, size_t workspace_bytes, int n, void *stream, const vppb200_rsgm_taps *taps, int phases,
                       int sets, int set, const vppb200_sgm_params *params, uint32_t uf, uint8_t *state_out = nullptr,
                       uint16_t *cost_out = nullptr, uint16_t *rival_out = nullptr)
{
    SgmParams prm;
    if (sgm_params_from(params, &prm)) return VPPB200_ERR_ARG;
    if (H <= 0 || W <= 0 || n <= 0 || (C != 1 && C != 3)) return VPPB200_ERR_ARG;
    if (D <= 0 || D % 8 != 0 || D > 256) return VPPB200_ERR_DISP;      // models/rsgm/rsgm.py:31-35
    if (phases <= 0 || phases > 7 || sets < 1 || sets > 4 || set < 0 || set >= sets) return VPPB200_ERR_ARG;
    const bool front = phases & VPPB200_PHASE_FRONT, mainp = phases & VPPB200_PHASE_MAIN, tail = phases & VPPB200_PHASE_TAIL;
    if (front && (!left || !left_vpp || !right_vpp)) return VPPB200_ERR_ARG;
    if (tail && !disp_out) return VPPB200_ERR_ARG;
    if ((hints == nullptr) != (validhints == nullptr)) return VPPB200_ERR_ARG;
    if (taps && phases != 7) return VPPB200_ERR_ARG;
    const RsgmDims d = make_dims(H, W, C, D);
    if (d.Hp < 8) return VPPB200_ERR_ARG;
    const bool info = state_out != nullptr;
    if (!workspace || workspace_bytes < rsgm_ws_layout(d, n, sets, 0, nullptr, nullptr, info)) return VPPB200_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    if (!rcp_lut) rcp_lut = device_rcp_lut(st);
    if (!rcp_lut) return cuda_fail("device_rcp_lut", cudaGetLastError());
    RsgmWs w;
    rsgm_ws_layout(d, n, sets, set, workspace, &w, info);
    int rc;
    StageMarks tm;
    if (phases == 7) tm.begin(st);                           // per-stage timing covers whole-pipeline calls only
    // the sweeps for parameters of their domain and shapes they hold (the layout of the cost volume follows: every phase of a batch
    // must see the same parameters and hints); otherwise the saturating per-path kernel, exact for any parameters
    const bool tiled = sweep_params_supported(prm, hints == nullptr) && aggregate_tile_supported(d.Wp, d.Hp, D, n);
    const bool want_volume = taps && taps->dsi_agg;          // only the test tap needs the aggregated volume itself
    const uint16_t *S_final = w.S;
    if (front) {
        // rsgm.py:258-262  pad (BORDER_REFLECT) + RGB2GRAY; the P2 guide is the raw byte stream of the padded `left`
        cudaStream_t side = side_stream(0);
        if (!side) side = st;                                // no side stream: everything in order on the caller's stream
        if (side != st && (rc = stream_chain(st, side))) return rc;
        // pad + gray + census in one kernel per image (the gray image stays in shared memory); two kernels where that does not apply
        if ((rc = launch_census_fused(right_vpp, w.census_r, d, n, side)) < 0) return rc;
        if (rc == 1) {
            if ((rc = launch_pad_gray(right_vpp, w.gray_r, d, n, side))) return rc;
            if ((rc = launch_census(w.gray_r, w.census_r, d.Wp, d.Hp, n, side))) return rc;
        }
        if ((rc = launch_pad_flatbytes(left, w.guide, d, n, st))) return rc;
        tm.done(VPPB200_STAGE_PAD_GRAY);
        if ((rc = launch_census_fused(left_vpp, w.census_l, d, n, st)) < 0) return rc;
        if (rc == 1) {
            if ((rc = launch_pad_gray(left_vpp, w.gray_l, d, n, st))) return rc;
            if ((rc = launch_census(w.gray_l, w.census_l, d.Wp, d.Hp, n, st))) return rc;
        }
        if (side != st && (rc = stream_chain(side, st))) return rc;
        tm.done(VPPB200_STAGE_CENSUS);
        // rsgm.py:263-268  Hamming volume (+ optional guided modulation: in the same kernel on the tiled path)
        if (tiled) {
            if ((rc = launch_cost_tile(w.census_l, w.census_r, w.dsi, d.Wp, d.Hp, D, n, guide_ops(hints, validhints, d), st))) return rc;
        } else {
            if ((rc = launch_cost_u8(w.census_l, w.census_r, w.dsi, d.Wp, d.Hp, D, n, st))) return rc;
            if (hints && (rc = launch_guided_u8(w.dsi, hints, validhints, d, n, st))) return rc;
        }
        tm.done(VPPB200_STAGE_COST);
    }
    if (mainp) {
        // rsgm.py:270  8-path aggregation (the reference's effective parameters unless the caller passed its own);
        // rsgm.py:272-273  WTA left (+ equiangular sub-pixel) and right
        if (tiled) {
            const StageHook hook = {StageMarks::hook, &tm};
            if (!want_volume) {
                // the last sweep consumes the final S on the fly: WTA left (+ sub-pixel) and right come out of the aggregation
                if ((rc = launch_aggregate_tile(w.guide, w.dsi, w.S, w.halo, d.Wp, d.Hp, D, n, w.dl, w.dr, rcp_lut, hints == nullptr, prm, &hook,
                                                uf, st, w.cost, w.rival)))
                    return rc < 0 ? rc : VPPB200_ERR_ARG;
            } else {
                if ((rc = launch_aggregate_tile(w.guide, w.dsi, w.S, w.halo, d.Wp, d.Hp, D, n, nullptr, nullptr, nullptr, hints == nullptr, prm,
                                                &hook, UNIQ_OFF, st)))
                    return rc < 0 ? rc : VPPB200_ERR_ARG;
                if ((rc = launch_s_tile_to_xyd(w.S, w.S_xyd, d.Wp, d.Hp, D, n, st))) return rc;
                S_final = w.S_xyd;
                if ((rc = launch_wta_both_subpix(S_final, w.dl, w.dr, d.Wp, d.Hp, D, rcp_lut, n, uf, st, w.cost, w.rival))) return rc;
            }
        } else {
            if ((rc = launch_aggregate_generic(w.guide, w.dsi, w.S, d.Wp, d.Hp, D, prm, n, st))) return rc;
            tm.done(VPPB200_STAGE_SGM_H_BWD);                // the per-path fallback is booked on the last sweep's slot
            if ((rc = launch_wta_both_subpix(S_final, w.dl, w.dr, d.Wp, d.Hp, D, rcp_lut, n, uf, st, w.cost, w.rival))) return rc;
        }
        tm.done(VPPB200_STAGE_WTA);
    }
    if (tail) {
        cudaStream_t side = side_stream(1);
        if (!side) side = st;
        if (side != st && (rc = stream_chain(st, side))) return rc;
        if ((rc = launch_median(w.dr, w.drf, d.Wp, d.Hp, n, side))) return rc;
        if ((rc = launch_interp_clip(w.drf, d.Wp, d.Hp, n, side))) return rc;
        if ((rc = launch_median(w.dl, w.dlf, d.Wp, d.Hp, n, st))) return rc;
        if ((rc = info ? launch_interp_clip_info(w.dlf, d, n, state_out, st) : launch_interp_clip(w.dlf, d.Wp, d.Hp, n, st))) return rc;
        if (side != st && (rc = stream_chain(side, st))) return rc;
        tm.done(VPPB200_STAGE_MEDIAN_INTERP);
        // rsgm.py:275-292  crop, LR check, speckle filter, sub-pixel restore, background fill
        if ((rc = info ? launch_tail_info(w.dlf, w.drf, disp_out, d, flags & 1, w.tail, n, state_out, w.cost, w.rival, cost_out, rival_out, st)
                       : launch_tail(w.dlf, w.drf, disp_out, d, flags & 1, w.tail, n, st)))
            return rc;
        tm.done(VPPB200_STAGE_TAIL);
    }
    tm.end();
    if (taps) {
        const size_t np = (size_t)n * d.Hp * d.Wp;
        if (taps->census_l) VPP_CUDA_TRY(cudaMemcpyAsync(taps->census_l, w.census_l, np * 4, cudaMemcpyDeviceToDevice, st));
        if (taps->census_r) VPP_CUDA_TRY(cudaMemcpyAsync(taps->census_r, w.census_r, np * 4, cudaMemcpyDeviceToDevice, st));
        if (taps->dsi_agg) VPP_CUDA_TRY(cudaMemcpyAsync(taps->dsi_agg, S_final, np * D * 2, cudaMemcpyDeviceToDevice, st));
        if (taps->disp_l) VPP_CUDA_TRY(cudaMemcpyAsync(taps->disp_l, w.dlf, np * 4, cudaMemcpyDeviceToDevice, st));
        if (taps->disp_r) VPP_CUDA_TRY(cudaMemcpyAsync(taps->disp_r, w.drf, np * 4, cudaMemcpyDeviceToDevice, st));
    }
    return VPPB200_OK;
}

extern "C" int vppb200_compute_rsgm_tapped(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp,
                                           const float *hints, const float *validhints, float *disp_out, int H, int W, int C,
                                           int D, int flags, const float *rcp_lut, void *workspace, size_t workspace_bytes,
                                           int n, void *stream, const vppb200_rsgm_taps *taps)
{
    return rsgm_phases(left, left_vpp, right_vpp, hints, validhints, disp_out, H, W, C, D, flags, rcp_lut, workspace,
                       workspace_bytes, n, stream, taps, 7, 1, 0, nullptr, UNIQ_OFF);
}

extern "C" int vppb200_compute_rsgm(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp, const float *hints,
                                    const float *validhints, float *disp_out, int H, int W, int C, int D, int flags,
                                    const float *rcp_lut, void *workspace, size_t workspace_bytes, int n, void *stream)
{
    return rsgm_phases(left, left_vpp, right_vpp, hints, validhints, disp_out, H, W, C, D, flags, rcp_lut, workspace,
                       workspace_bytes, n, stream, nullptr, 7, 1, 0, nullptr, UNIQ_OFF);
}

extern "C" int vppb200_compute_rsgm_phases(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp,
                                           const float *hints, const float *validhints, float *disp_out, int H, int W, int C,
                                           int D, int flags, const float *rcp_lut, void *workspace, size_t workspace_bytes,
                                           int n, void *stream, int phases, int sets, int set)
{
    return rsgm_phases(left, left_vpp, right_vpp, hints, validhints, disp_out, H, W, C, D, flags, rcp_lut, workspace,
                       workspace_bytes, n, stream, nullptr, phases, sets, set, nullptr, UNIQ_OFF);
}

extern "C" int vppb200_compute_rsgm_ex(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp, const float *hints,
                                       const float *validhints, float *disp_out, int H, int W, int C, int D, int flags,
                                       const float *rcp_lut, void *workspace, size_t workspace_bytes, int n, void *stream, int phases,
                                       int sets, int set, const vppb200_rsgm_taps *taps, const vppb200_sgm_params *params)
{
    return rsgm_phases(left, left_vpp, right_vpp, hints, validhints, disp_out, H, W, C, D, flags, rcp_lut, workspace,
                       workspace_bytes, n, stream, taps, phases, sets, set, params, UNIQ_OFF);
}

extern "C" int vppb200_compute_rsgm_uniq(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp, const float *hints,
                                         const float *validhints, float *disp_out, int H, int W, int C, int D, int flags,
                                         const float *rcp_lut, void *workspace, size_t workspace_bytes, int n, void *stream,
                                         int phases, int sets, int set, const vppb200_rsgm_taps *taps,
                                         const vppb200_sgm_params *params, float uniqueness)
{
    uint32_t uf;
    const int rc = uniq_factor(uniqueness, &uf);
    if (rc) return rc;
    return rsgm_phases(left, left_vpp, right_vpp, hints, validhints, disp_out, H, W, C, D, flags, rcp_lut, workspace,
                       workspace_bytes, n, stream, taps, phases, sets, set, params, uf);
}

extern "C" size_t vppb200_rsgm_info_workspace_bytes(int H, int W, int C, int D, int n, int sets)
{
    if (H <= 0 || W <= 0 || n <= 0 || D <= 0 || D % 8 || D > 256 || (C != 1 && C != 3) || sets < 1 || sets > 4) return 0;
    return rsgm_ws_layout(make_dims(H, W, C, D), n, sets, 0, nullptr, nullptr, true);
}

extern "C" int vppb200_compute_rsgm_info(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp, const float *hints,
                                         const float *validhints, float *disp_out, int H, int W, int C, int D, int flags,
                                         const float *rcp_lut, void *workspace, size_t workspace_bytes, int n, void *stream,
                                         int phases, int sets, int set, const vppb200_rsgm_taps *taps,
                                         const vppb200_sgm_params *params, float uniqueness, uint8_t *state_out, uint16_t *cost_out,
                                         uint16_t *rival_out)
{
    uint32_t uf;
    const int rc = uniq_factor(uniqueness, &uf);
    if (rc) return rc;
    if (!state_out || !cost_out || !rival_out) return VPPB200_ERR_ARG;
    return rsgm_phases(left, left_vpp, right_vpp, hints, validhints, disp_out, H, W, C, D, flags, rcp_lut, workspace,
                       workspace_bytes, n, stream, taps, phases, sets, set, params, uf, state_out, cost_out, rival_out);
}

extern "C" int vppb200_sgm_params_fast(const vppb200_sgm_params *params, int guided)
{
    SgmParams prm;
    if (sgm_params_from(params, &prm)) return VPPB200_ERR_ARG;
    return sweep_params_supported(prm, !guided) ? 1 : 0;
}

// ---- one frame split into row bands over several GPUs (SURVEY.md 8e rows 2 and 5) ------------------------------
// The stages of compute_rsgm as three calls, so that a caller (vppstereo_b200/banded.py) can run the aggregation of a band on
// each GPU and hand the vertical sweeps' row state from band to band:
//   front_census: pad + gray + census of the WHOLE frame (a few MB; every rank does it) -> guide, census_l, census_r
//   sgm_band:     Hamming volume and the four sweeps for rows [row0, row0 + rows) only (the 2.2 GB of a Middlebury frame's
//                 volumes are what is split), raw left / right disparities of those rows out
//   tail:         median .. background fill on the gathered raw disparities of the whole frame
namespace vppb200 {
struct BandWs { uint8_t *gray_l, *gray_r; void *halo; float *dlf, *drf; TailBufs tail; };
static size_t band_ws_layout(const RsgmDims &d, int rows, void *base, BandWs *ws)
{
    size_t off = 0;
    char *b = (char *)base;
    auto take = [&](size_t bytes) { size_t o = off; off += align256(bytes); return b ? b + o : (char *)nullptr; };
    const size_t np = (size_t)d.Hp * d.Wp, nc = (size_t)d.H * tail_stride(d.W);
    BandWs w;
    w.gray_l = (uint8_t *)take(np); w.gray_r = (uint8_t *)take(np);
    w.halo = (void *)take(sweep_halo_bytes(d.Wp, rows > 0 ? rows : d.Hp, d.D, 1));
    w.dlf = (float *)take(np * 4); w.drf = (float *)take(np * 4);
    w.tail.u8 = (uint8_t *)take(nc); w.tail.label = (int *)take(nc * 4); w.tail.count = (int *)take(nc * 4);
    if (ws) *ws = w;
    return off;
}
}  // namespace vppb200

extern "C" size_t vppb200_banded_workspace_bytes(int H, int W, int C, int D)
{
    if (H <= 0 || W <= 0 || D <= 0 || D % 8 || D > 256 || (C != 1 && C != 3)) return 0;
    return band_ws_layout(make_dims(H, W, C, D), 0, nullptr, nullptr);
}

extern "C" int vppb200_banded_dims(int H, int W, int C, int D, int *Hp, int *Wp, int64_t *state_words, int64_t *volume_bytes_per_row)
{
    if (H <= 0 || W <= 0 || D <= 0 || D % 8 || D > 256 || (C != 1 && C != 3)) return VPPB200_ERR_ARG;
    const RsgmDims d = make_dims(H, W, C, D);
    if (Hp) *Hp = d.Hp;
    if (Wp) *Wp = d.Wp;
    if (state_words) *state_words = sweep_state_words(d.Wp, D);
    if (volume_bytes_per_row) *volume_bytes_per_row = (int64_t)(tile_volume_elems(d.Wp, 1, D, 1));      // uint8 costs; S = 2x
    return VPPB200_OK;
}

extern "C" int vppb200_rsgm_front_census(const uint8_t *left, const uint8_t *left_vpp, const uint8_t *right_vpp, uint8_t *guide,
                                         uint32_t *census_l, uint32_t *census_r, int H, int W, int C, int D, void *workspace,
                                         size_t workspace_bytes, void *stream)
{
    if (!left || !left_vpp || !right_vpp || !guide || !census_l || !census_r || H <= 0 || W <= 0 || (C != 1 && C != 3)) return VPPB200_ERR_ARG;
    if (D <= 0 || D % 8 != 0 || D > 256) return VPPB200_ERR_DISP;
    const RsgmDims d = make_dims(H, W, C, D);
    if (!workspace || workspace_bytes < band_ws_layout(d, 0, nullptr, nullptr)) return VPPB200_ERR_WORKSPACE;
    BandWs w;
    band_ws_layout(d, 0, workspace, &w);
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if ((rc = launch_pad_gray(right_vpp, w.gray_r, d, 1, st))) return rc;
    if ((rc = launch_census(w.gray_r, census_r, d.Wp, d.Hp, 1, st))) return rc;
    if ((rc = launch_pad_gray(left_vpp, w.gray_l, d, 1, st))) return rc;
    if ((rc = launch_pad_flatbytes(left, guide, d, 1, st))) return rc;
    return launch_census(w.gray_l, census_l, d.Wp, d.Hp, 1, st);
}

extern "C" int vppb200_sgm_band_uniq(const uint8_t *guide, const uint32_t *census_l, const uint32_t *census_r, uint8_t *cost_band,
                                     uint16_t *S_band, int H, int W, int C, int D, int row0, int rows, int phases,
                                     const uint32_t *state_in, uint32_t *state_out, float *dl_band, float *dr_band,
                                     const float *rcp_lut, void *workspace, size_t workspace_bytes, void *stream,
                                     const vppb200_sgm_params *params, const float *hints, const float *validhints, float uniqueness)
{
    uint32_t uf;
    if (uniq_factor(uniqueness, &uf)) return VPPB200_ERR_UNIQUENESS;
    SgmParams prm;
    if (sgm_params_from(params, &prm)) return VPPB200_ERR_ARG;
    if ((hints == nullptr) != (validhints == nullptr)) return VPPB200_ERR_ARG;
    const bool plain = hints == nullptr;
    if (!sweep_params_supported(prm, plain)) return VPPB200_ERR_ARG;     // bands exist on the sweeps only
    if (!guide || !cost_band || !S_band || H <= 0 || W <= 0 || (C != 1 && C != 3) || phases <= 0 || phases > 31) return VPPB200_ERR_ARG;
    if (D <= 0 || D % 8 != 0 || D > 256) return VPPB200_ERR_DISP;
    if ((phases & 1) && (!census_l || !census_r)) return VPPB200_ERR_ARG;
    if ((phases & 16) && (!dl_band || !dr_band)) return VPPB200_ERR_ARG;
    const RsgmDims d = make_dims(H, W, C, D);
    if (!workspace || workspace_bytes < band_ws_layout(d, 0, nullptr, nullptr)) return VPPB200_ERR_WORKSPACE;
    BandWs w;
    band_ws_layout(d, 0, workspace, &w);
    cudaStream_t st = (cudaStream_t)stream;
    if (!rcp_lut) rcp_lut = device_rcp_lut(st);
    if (!rcp_lut) return cuda_fail("device_rcp_lut", cudaGetLastError());
    return launch_aggregate_band(guide, census_l, census_r, cost_band, S_band, w.halo, d.Wp, d.Hp, D, row0, rows, 1, phases, state_in,
                                 state_out, dl_band, dr_band, rcp_lut, plain, prm, guide_ops(hints, validhints, d), uf, st);
}

extern "C" int vppb200_sgm_band_guided(const uint8_t *guide, const uint32_t *census_l, const uint32_t *census_r, uint8_t *cost_band,
                                       uint16_t *S_band, int H, int W, int C, int D, int row0, int rows, int phases,
                                       const uint32_t *state_in, uint32_t *state_out, float *dl_band, float *dr_band,
                                       const float *rcp_lut, void *workspace, size_t workspace_bytes, void *stream,
                                       const vppb200_sgm_params *params, const float *hints, const float *validhints)
{
    return vppb200_sgm_band_uniq(guide, census_l, census_r, cost_band, S_band, H, W, C, D, row0, rows, phases, state_in, state_out,
                                 dl_band, dr_band, rcp_lut, workspace, workspace_bytes, stream, params, hints, validhints, 1.0f);
}

extern "C" int vppb200_sgm_band_ex(const uint8_t *guide, const uint32_t *census_l, const uint32_t *census_r, uint8_t *cost_band,
                                   uint16_t *S_band, int H, int W, int C, int D, int row0, int rows, int phases, const uint32_t *state_in,
                                   uint32_t *state_out, float *dl_band, float *dr_band, const float *rcp_lut, void *workspace,
                                   size_t workspace_bytes, void *stream, const vppb200_sgm_params *params)
{
    return vppb200_sgm_band_guided(guide, census_l, census_r, cost_band, S_band, H, W, C, D, row0, rows, phases, state_in, state_out,
                                   dl_band, dr_band, rcp_lut, workspace, workspace_bytes, stream, params, nullptr, nullptr);
}

extern "C" int vppb200_sgm_band(const uint8_t *guide, const uint32_t *census_l, const uint32_t *census_r, uint8_t *cost_band,
                                uint16_t *S_band, int H, int W, int C, int D, int row0, int rows, int phases, const uint32_t *state_in,
                                uint32_t *state_out, float *dl_band, float *dr_band, const float *rcp_lut, void *workspace,
                                size_t workspace_bytes, void *stream)
{
    return vppb200_sgm_band_ex(guide, census_l, census_r, cost_band, S_band, H, W, C, D, row0, rows, phases, state_in, state_out,
                               dl_band, dr_band, rcp_lut, workspace, workspace_bytes, stream, nullptr);
}

extern "C" int vppb200_rsgm_tail(float *dl, float *dr, float *disp_out, int H, int W, int C, int D, int flags, void *workspace,
                                 size_t workspace_bytes, void *stream)
{
    if (!dl || !dr || !disp_out || H <= 0 || W <= 0 || (C != 1 && C != 3)) return VPPB200_ERR_ARG;
    if (D <= 0 || D % 8 != 0 || D > 256) return VPPB200_ERR_DISP;
    const RsgmDims d = make_dims(H, W, C, D);
    if (!workspace || workspace_bytes < band_ws_layout(d, 0, nullptr, nullptr)) return VPPB200_ERR_WORKSPACE;
    BandWs w;
    band_ws_layout(d, 0, workspace, &w);
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if ((rc = launch_median(dr, w.drf, d.Wp, d.Hp, 1, st))) return rc;
    if ((rc = launch_interp_clip(w.drf, d.Wp, d.Hp, 1, st))) return rc;
    if ((rc = launch_median(dl, w.dlf, d.Wp, d.Hp, 1, st))) return rc;
    if ((rc = launch_interp_clip(w.dlf, d.Wp, d.Hp, 1, st))) return rc;
    return launch_tail(w.dlf, w.drf, disp_out, d, flags & 1, w.tail, 1, st);
}

// ---- hand-off to the networks (test.py:179-197) -----------------------------------------------------------
namespace vppb200 {
__global__ void u8hwc_to_f32chw_kernel(const uint8_t *__restrict__ src, float *__restrict__ dst, int H, int W, int C, int pt,
                                       int pl, int Ho, int Wo, long total)
{
    long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int x = (int)(t % Wo), y = (int)((t / Wo) % Ho), c = (int)((t / ((long)Wo * Ho)) % C);
    const long f = t / ((long)Wo * Ho * C);
    const int sy = min(max(y - pt, 0), H - 1), sx = min(max(x - pl, 0), W - 1);       // replicate
    const uint8_t v = src[((f * H + sy) * W + sx) * C + c];
    dst[t] = (float)__ddiv_rn((double)v, 255.0);                                       // float32(u8 / 255.0)
}

// (255 * im).astype(np.uint8) of a [C,H,W] float32 image in HWC order (test.py:158-159,:210-212): float32 product, truncation
__global__ void f32chw_to_u8hwc_kernel(const float *__restrict__ src, uint8_t *__restrict__ dst, int H, int W, int C, long total)
{
    long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int c = (int)(t % C), x = (int)((t / C) % W), y = (int)((t / ((long)C * W)) % H);
    const long f = t / ((long)C * W * H);
    const float v = __fmul_rn(255.0f, src[((f * C + c) * H + y) * W + x]);
    dst[t] = (uint8_t)(int)v;                       // values are in [0, 255]; the reference's cast is undefined outside
}
}  // namespace vppb200

extern "C" int vppb200_f32chw_to_u8hwc(const float *src, uint8_t *dst, int H, int W, int C, int n, void *stream)
{
    if (!src || !dst || H <= 0 || W <= 0 || C <= 0 || n <= 0) return VPPB200_ERR_ARG;
    const long total = (long)n * C * H * W;
    f32chw_to_u8hwc_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(src, dst, H, W, C, total);
    VPP_LAUNCH_CHECK("f32chw_to_u8hwc_kernel");
    return VPPB200_OK;
}

extern "C" int vppb200_u8hwc_to_f32chw(const uint8_t *src, float *dst, int H, int W, int C, int pad_top, int pad_bottom,
                                       int pad_left, int pad_right, int n, void *stream)
{
    if (!src || !dst || H <= 0 || W <= 0 || C <= 0 || n <= 0 || pad_top < 0 || pad_bottom < 0 || pad_left < 0 || pad_right < 0)
        return VPPB200_ERR_ARG;
    const int Ho = H + pad_top + pad_bottom, Wo = W + pad_left + pad_right;
    const long total = (long)n * C * Ho * Wo;
    u8hwc_to_f32chw_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(src, dst, H, W, C, pad_top, pad_left, Ho, Wo, total);
    VPP_LAUNCH_CHECK("u8hwc_to_f32chw_kernel");
    return VPPB200_OK;
}
