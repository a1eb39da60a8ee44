// mapf_capi.cu -- C ABI (include/mapf_b200.h) over the sm_100a kernels: context creation, host-side derivation of
// the env constants in the reference's floating-point order, kernel dispatch.
//
// Reference citations are file:line relative to /root/reference/gym_mapf/envs/.
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <vector>

#include "../../include/mapf_b200.h"
#include "mapf_host.h"
#include "mapf_kernels.cuh"

typedef unsigned __int128 u128;

// ---------------------------------------------------------------------------------------------------------------
// error reporting
// ---------------------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                                         \
    do {                                                                                                       \
        cudaError_t _e = (expr);                                                                               \
        if (_e != cudaSuccess) return fail(MAPF_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(_e),     \
                                           __FILE__, __LINE__);                                                \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
};

// ---------------------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------------------
#define MAPF_HOST_STREAMS 2   // mapf_step_host: the staged path pipelines two halves
struct mapf_ctx {
    DevSpec sp;
    mapf_info info;
    int device = 0;
    int threads = 256;           // CTA size of the hot kernels
    int threads_expand = 256;    // ... of k_expand (wider for many agents)
    size_t smem_base = 0;        // small tables + staged move table
    size_t smem_expand = 0;      // smem_base + per-warp expand slabs
    size_t smem_backup = 0;      // smem_base + per-warp backup slabs
    int threads_step = 0;  // CTA size of k_step (ks.step_threads, else `threads`)
    int grid_step1 = 0, grid_step2 = 0, grid_step_tape = 0, grid_rollout = 0, grid_rollout2 = 0, grid_rollout_tape = 0;
    int grid_expand = 0, grid_expand_range = 0, grid_plain = 0, grid_backup = 0, grid_backup_range = 0;
    int grid_evaluate[4] = {0, 0, 0, 0};  // k_evaluate / k_evaluate_groups by policy kind
    int grid_rtdp = 0, grid_evaluate_table = 0;
    KernelSet ks;
    u32 pat_triple[MAPF_MAX_PATTERNS];  // merge patterns (see PatternList)
    int n_patterns = 0;
    double probtab[8];                  // probability of a merged outcome, indexed by its candidate mask
    bool philox_ok = true;              // every pattern's probabilities add up to 1: device-side sampling is exact
    PatternTables pt;                   // host copy of the per-pattern tables (the device copy is in the image)
    unsigned char *d_image = nullptr;   // DevSpec::image; the move table is its tail
    u64 *d_lut = nullptr;               // = d_image + (MAPF_SMEM_LUT - MAPF_SMEM_IMG)
    u32 *d_cell_rc = nullptr, *d_colbits = nullptr, *d_colbase = nullptr;
    std::vector<u64> h_lut;
    std::vector<u32> h_cell_rc;
    // mapf_step_host staging
    std::mutex mu;
    cudaStream_t hs[MAPF_HOST_STREAMS] = {};
    unsigned char *d_stage = nullptr;
    size_t d_stage_bytes = 0;
    unsigned char *h_small = nullptr;   // page-locked scratch of the small-batch host step (mapped into the device)
    unsigned char *h_small_dev = nullptr;
};

static bool pick_kernels(int n, int words, bool luts, KernelSet *ks) {
#ifdef MAPF_ONLY_N  // experiment builds (tools/sweep_step.py): a single agent count
#define CAT2_(a, b) a##b
#define CAT2(a, b) CAT2_(a, b)
    static mapf_kernels_fn table[MAPF_MAXN + 1] = {nullptr};
    table[MAPF_ONLY_N] = CAT2(mapf_get_kernels_, MAPF_ONLY_N);
    if (n != MAPF_ONLY_N) return false;
#else
    static const mapf_kernels_fn table[MAPF_MAXN + 1] = {
        nullptr, mapf_get_kernels_1, mapf_get_kernels_2, mapf_get_kernels_3, mapf_get_kernels_4, mapf_get_kernels_5,
        mapf_get_kernels_6, mapf_get_kernels_7, mapf_get_kernels_8, mapf_get_kernels_9, mapf_get_kernels_10,
        mapf_get_kernels_11, mapf_get_kernels_12, mapf_get_kernels_13};
#endif
    if (n < 1 || n > MAPF_MAXN) return false;
    table[n](words, luts ? 1 : 0, ks);
    return ks->step_tape != nullptr;
}

static FastDiv make_fastdiv(u64 d) {
    // branch-free form: q = mulhi(x, magic); q = (((x - q) >> 1) + q) >> shift, exact for every 64-bit x
    FastDiv f;
    f.magic = 0; f.shift = 0; f.pad = 0;
    if (d <= 1) return f;  // x >> 1 >> ... is never taken: d == 1 only occurs when every state is 0
    const int fl = 63 - __builtin_clzll(d);
    if ((d & (d - 1)) == 0) { f.shift = (u32)(fl - 1); return f; }  // magic 0: ((x >> 1) >> (fl - 1))
    const u128 num = (u128)1 << (64 + fl);
    u64 proposed = (u64)(num / d);
    const u64 rem = (u64)(num % d);
    proposed += proposed;
    const u64 twice = rem + rem;
    if (twice >= d || twice < rem) proposed += 1;
    f.magic = proposed + 1;
    f.shift = (u32)fl;
    return f;
}

static Div32 make_div32(u32 d) {
    // The dividend is a two-digit chunk x < d*d.  Round-up magic m = ceil(2**s / d): umulhi(x, m) >> (s - 32) is
    // exact when (m*d - 2**s) * (d*d - 1) < 2**s; take the smallest s >= 32 with m < 2**32 that satisfies it.
    Div32 f;
    f.pad = 0;
    if (d <= 1) { f.magic = 0; f.shift = 0; f.fix = 0; return f; }  // x is always 0
    const u128 xmax = (u128)d * d - 1;
    for (int s = 32; s < 64; ++s) {
        const u128 p = (u128)1 << s;
        const u128 m = (p + d - 1) / d;
        if (m >> 32) break;
        const u128 e = m * d - p;
        if (e * xmax < p) { f.magic = (u32)m; f.shift = (u32)(s - 32); f.fix = 0; return f; }
    }
    // round-DOWN magic: floor(x / d) or one less for every 32-bit x; the kernels fix it with one compare
    const int fl = 31 - __builtin_clz(d);
    f.shift = (u32)fl;
    const u64 p = 1ull << (32 + fl);
    const u64 m = p / d;
    f.magic = (u32)(m > 0xffffffffull ? 0xffffffffull : m);
    f.fix = 1;
    return f;
}

extern "C" const char *mapf_last_error(void) { return g_err; }
extern "C" const char *mapf_version(void) { return "mapf_b200 0.1 (sm_100a)"; }

extern "C" void mapf_ctx_destroy(mapf_ctx *ctx) {
    if (!ctx) return;
    {
        DeviceGuard g(ctx->device);
        cudaFree(ctx->d_image);
        cudaFree(ctx->d_cell_rc);
        cudaFree(ctx->d_colbits);
        cudaFree(ctx->d_colbase);
        cudaFree(ctx->d_stage);
        if (ctx->h_small) cudaFreeHost(ctx->h_small);
        for (int i = 0; i < MAPF_HOST_STREAMS; ++i)
            if (ctx->hs[i]) cudaStreamDestroy(ctx->hs[i]);
    }
    delete ctx;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a cap PER FUNCTION, and the kernel functions are shared by every
// context with the same (agents, words, staged): keep a running maximum per (device, function) and never lower it -- a
// later, smaller context would otherwise shrink the cap under an earlier, larger one and its launches would fail.
static int raise_smem_cap(int device, const void *fn, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<int, const void *>, size_t> cap;
    std::lock_guard<std::mutex> lock(mu);
    size_t &cur = cap[std::make_pair(device, fn)];
    if (bytes <= cur || bytes <= 48 * 1024) return MAPF_OK;
    CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    cur = bytes;
    return MAPF_OK;
}

static int occupancy_grid(const void *fn, int threads, size_t smem, int sm_count, int *grid) {
    int per_sm = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, smem));
    if (per_sm < 1) return fail(MAPF_ERR_CUDA, "kernel does not fit on an SM (threads=%d smem=%zu)", threads, smem);
    *grid = per_sm * sm_count;
    return MAPF_OK;
}

// Every first-occurrence merge of the candidates that have positive probability (mapf_env.py:172-182), as
// 9-bit mask triples; at most 5 exist (the set partitions of three candidates).
static int enumerate_patterns(int cand_mask, u32 *triples) {
    int count = 0;
    for (int labels = 0; labels < 27; ++labels) {
        int lab[3] = {labels % 3, (labels / 3) % 3, labels / 9};
        u32 mask[3] = {0, 0, 0};
        int dest[3] = {-1, -1, -1}, k = 0;
        for (int j = 0; j < 3; ++j) {
            if (!((cand_mask >> j) & 1)) continue;
            int at = -1;
            for (int q = 0; q < k; ++q)
                if (dest[q] == lab[j] && at < 0) at = q;
            if (at >= 0) mask[at] |= 1u << j;
            else { dest[k] = lab[j]; mask[k] = 1u << j; ++k; }
        }
        const u32 t = mask[0] | (mask[1] << 3) | (mask[2] << 6);
        bool seen = false;
        for (int q = 0; q < count; ++q) seen = seen || triples[q] == t;
        if (!seen && count < MAPF_MAX_PATTERNS) triples[count++] = t;
    }
    return count;
}

extern "C" int mapf_ctx_create(const mapf_spec *spec, int device, mapf_ctx **out) {
    if (!spec || !out || !spec->obstacles || !spec->start_rc || !spec->goal_rc)
        return fail(MAPF_ERR_INVALID, "mapf_ctx_create: NULL argument");
    *out = nullptr;
    const int H = spec->height, W = spec->width, n = spec->n_agents;
    if (H < 1 || W < 1) return fail(MAPF_ERR_INVALID, "empty grid");
    if (n < 1 || n > MAPF_MAX_AGENTS)
        return fail(MAPF_ERR_UNSUPPORTED, "%d agents: this build supports 1..%d", n, MAPF_MAX_AGENTS);
    if (spec->criterion != MAPF_SOC && spec->criterion != MAPF_MAKESPAN)
        return fail(MAPF_ERR_INVALID, "unknown optimisation criterion %d", spec->criterion);
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev < 1 || device < 0 || device >= n_dev)
        return fail(MAPF_ERR_NO_DEVICE, "CUDA device %d is not available (%d devices): there is no CPU fallback",
                    device, n_dev);

    // ---- column-major free-cell numbering (grid.py:37-40, mapf_env.py:142-143) and the column bitmap
    const int wpc = (H + 31) / 32;
    std::vector<u32> colbits((size_t)W * wpc, 0u), colbase(W, 0u);
    std::vector<int> id_of((size_t)H * W, -1);
    int L = 0;
    for (int c = 0; c < W; ++c) {
        colbase[c] = (u32)L;
        for (int r = 0; r < H; ++r)
            if (!spec->obstacles[(size_t)r * W + c]) {
                colbits[(size_t)c * wpc + (r >> 5)] |= 1u << (r & 31);
                id_of[(size_t)r * W + c] = L++;
            }
    }
    if (L < 1) return fail(MAPF_ERR_INVALID, "the grid has no free cell");
    if (L > MAPF_MAX_CELLS) return fail(MAPF_ERR_UNSUPPORTED, "%d free cells: this build supports up to %d", L,
                                        MAPF_MAX_CELLS);

    mapf_ctx *ctx = new (std::nothrow) mapf_ctx();
    if (!ctx) return fail(MAPF_ERR_INVALID, "out of host memory");
    ctx->device = device;
    DevSpec &sp = ctx->sp;
    memset(&sp, 0, sizeof(sp));
    memset(&ctx->pt, 0, sizeof(ctx->pt));
    sp.n = n; sp.L = L; sp.H = H; sp.Wd = W;
    sp.soc = spec->criterion == MAPF_SOC ? 1 : 0;

    // ---- starts / goals must be free cells: the reference raises KeyError (mapf_env.py:155,158,369)
    int start_id[MAPF_MAXN], goal_id[MAPF_MAXN];
    for (int i = 0; i < n; ++i) {
        const int sr = spec->start_rc[2 * i], sc = spec->start_rc[2 * i + 1];
        const int gr = spec->goal_rc[2 * i], gc = spec->goal_rc[2 * i + 1];
        if (sr < 0 || sr >= H || sc < 0 || sc >= W || id_of[(size_t)sr * W + sc] < 0) {
            delete ctx;
            return fail(MAPF_ERR_KEY, "(%d, %d)", sr, sc);
        }
        if (gr < 0 || gr >= H || gc < 0 || gc >= W || id_of[(size_t)gr * W + gc] < 0) {
            delete ctx;
            return fail(MAPF_ERR_KEY, "(%d, %d)", gr, gc);
        }
        start_id[i] = id_of[(size_t)sr * W + sc];
        goal_id[i] = id_of[(size_t)gr * W + gc];
        sp.start[i] = (u16)start_id[i];
        sp.goal[i] = (u16)goal_id[i];
    }

    // ---- nS = L**n, nA = 5**n (mapf_env.py:145-146); state width
    u128 nS = 1;
    for (int i = 0; i < n; ++i) {
        if (nS > (((u128)1 << 127) / (u128)L)) {
            delete ctx;
            return fail(MAPF_ERR_UNSUPPORTED, "L**n = %d**%d does not fit 127 bits", L, n);
        }
        nS *= (u128)L;
    }
    sp.words = nS < ((u128)1 << 63) ? 1 : 2;
    sp.smax[0] = (u64)(nS - 1); sp.smax[1] = (u64)((nS - 1) >> 64);
    u64 nA = 1;
    for (int i = 0; i < n; ++i) nA *= 5;
    sp.nA = nA;
    // decode plan: two digits (radix L*L < 2**32) per 64-bit division
    {
        const u64 ll = (u64)L * (u64)L;
        sp.LL = (u32)ll;
        sp.divLL = make_fastdiv(ll);
        // reciprocals rounded UP (checked exactly in 128-bit integers: inv = m * 2**e with a 53-bit m), see fdiv_floor()
        auto recip_up = [](u64 d) {
            double inv = 1.0 / (double)d;
            for (;;) {
                int e;
                const double m = frexp(inv, &e);              // inv = m * 2**e, 0.5 <= m < 1
                const u64 mi = (u64)ldexp(m, 53);              // 53-bit integer mantissa
                // inv * d >= 1  <=>  mi * d >= 2**(53 - e)
                const u128 lhs = (u128)mi * (u128)d;
                const int sh = 53 - e;
                if (sh < 127 && lhs >= ((u128)1 << sh)) return inv;
                inv = nextafter(inv, 2.0);
            }
        };
        sp.invLL_up = recip_up(ll);
        sp.negcLL = -ldexp(sp.invLL_up, 52);
        sp.invL_up = recip_up((u64)L);
        sp.negcL = -ldexp(sp.invL_up, 52);
        sp.negLL = (u32)(0u - (u32)ll);
        sp.negL = (u32)(0u - (u32)L);
        // expand with cached head agents (see HeadCache): tail = last six agents
        sp.head_ok = 0;
        sp.powLH = 1;
        if (n >= EXPAND_HEAD_MIN_AGENTS) {
            u128 t6 = 1, th = 1;
            for (int i = 0; i < EXPAND_TAIL_AGENTS; ++i) t6 *= (u128)L;
            bool fits = t6 < ((u128)1 << 63);
            for (int i = 0; i < n - EXPAND_TAIL_AGENTS; ++i) { th *= (u128)L; fits = fits && th < ((u128)1 << 63); }
            if (fits) { sp.head_ok = 1; sp.powLH = (u64)th; }
        }
        // two-word states: split point of the decode / encode (see DevSpec::split_ok)
        sp.split_ok = 0;
        if (sp.words == 2 && n >= 2) {
            const int klo = MAPF_SPLIT_KLO(n) < n ? MAPF_SPLIT_KLO(n) : n - 1;
            u128 D = 1, hi_span = 1;
            bool fits = true;
            for (int i = 0; i < klo; ++i) { D *= (u128)L; fits = fits && D < ((u128)1 << 63); }
            for (int i = klo; i < n; ++i) { hi_span *= (u128)L; fits = fits && hi_span < ((u128)1 << 49); }
            if (fits) {
                sp.split_ok = 1;
                sp.splitD = (u64)D;
                sp.invD = 1.0 / (double)(u64)D;
            }
        }
        sp.divL = make_div32((u32)L);
        u128 v = nS - 1;
        for (int pass = 0; pass < 8; ++pass) {
            int limbs = 1;
            for (int w = 3; w >= 1; --w)
                if ((v >> (32 * w)) != 0) { limbs = w + 1; break; }
            sp.limbs[pass] = limbs;
            v /= (u128)ll;
        }
    }
    u128 s0 = 0, sg = 0, mul = 1;
    for (int i = 0; i < n; ++i) {  // vector_to_integer (__init__.py:70-79)
        s0 += (u128)start_id[i] * mul;
        sg += (u128)goal_id[i] * mul;
        mul *= (u128)L;
    }
    sp.s0_terminal = s0 == sg ? 1 : 0;  // is_terminal(starts) (mapf_env.py:210-223): every agent on its goal ...
    for (int i = 0; i < n; ++i)
        for (int j = i + 1; j < n; ++j)
            if (start_id[i] == start_id[j]) sp.s0_terminal = 1;  // ... or two agents on one cell
    sp.s0[0] = (u64)s0; sp.s0[1] = (u64)(s0 >> 64);
    sp.sgoal[0] = (u64)sg; sp.sgoal[1] = (u64)(sg >> 64);

    // ---- probabilities in the reference's order (mapf_env.py:131-132,168-170,177-179)
    const double rf = spec->fail_prob / 2, lf = spec->fail_prob / 2;
    const double cand[3] = {1 - rf - lf, rf, lf};
    sp.cand_mask = 0;
    for (int j = 0; j < 3; ++j)
        if (cand[j] > 0) sp.cand_mask |= 1 << j;
    if (sp.cand_mask == 0) {
        delete ctx;
        return fail(MAPF_ERR_INVALID, "fail_prob %g leaves no outcome with positive probability", spec->fail_prob);
    }
    ctx->probtab[0] = 0.0;
    for (int m = 1; m < 8; ++m) {  // a merged outcome's probability: its candidates added in list order
        double s = 0.0;
        bool first = true;
        for (int j = 0; j < 3; ++j)
            if ((m >> j) & 1) { s = first ? cand[j] : s + cand[j]; first = false; }
        ctx->probtab[m] = s;
    }
    ctx->n_patterns = enumerate_patterns(sp.cand_mask, ctx->pat_triple);
    for (int p = 0; p < ctx->n_patterns; ++p) {
        double acc = 0.0;
        for (int j = 0; j < 3; ++j) {
            const u32 m = (ctx->pat_triple[p] >> (3 * j)) & 7u;
            const double pj = ctx->probtab[m];
            ctx->pt.pp[p][j] = pj;
            if (m) acc = j == 0 ? pj : acc + pj;  // np.cumsum: sequential fp64 adds (mapf_env.py:255)
            ctx->pt.cum[p][j] = acc;
            // largest 32-bit w with acc > w * 2**-32, i.e. w < acc * 2**32 (an exact scaling)
            double x = ceil(acc * 4294967296.0);
            if (x > 4294967296.0) x = 4294967296.0;
            if (x < 1.0) x = 1.0;  // cannot happen: the first merged outcome has positive probability
            ctx->pt.thr[p][j] = ~(u32)((u64)x - 1);  // stored complemented, see count_below()
        }
        // the device-side sampling mode counts thresholds below the draw, which needs the pattern's last
        // cumulative probability to reach 1 (within 2**-32): true whenever right_fail + left_fail <= 1
        const int k = (ctx->pat_triple[p] & 7u ? 1 : 0) + ((ctx->pat_triple[p] >> 3) & 7u ? 1 : 0) +
                      ((ctx->pat_triple[p] >> 6) & 7u ? 1 : 0);
        if (ctx->pt.thr[p][k - 1] != 0u) ctx->philox_ok = false;  // ~(2**32 - 1)
    }
    // ---- rewards (mapf_env.py:225-235, 436-446), one entry per number of parked agents
    for (int k = 0; k <= n; ++k) {
        const double live = sp.soc ? (double)(n - k) * spec->reward_of_living : spec->reward_of_living;
        ctx->pt.reward[0 * MAPF_REW_STRIDE + k] = live;
        ctx->pt.reward[1 * MAPF_REW_STRIDE + k] = spec->reward_of_clash + live;
        ctx->pt.reward[2 * MAPF_REW_STRIDE + k] = spec->reward_of_goal + live;
        ctx->pt.reward[3 * MAPF_REW_STRIDE + k] = 0.0;  // step from a terminal state (mapf_env.py:240)
    }

    // ---- device side
    DeviceGuard guard(device);
    if (!guard.ok) { delete ctx; return fail(MAPF_ERR_CUDA, "cannot select device %d", device); }
    cudaDeviceProp prop;
    cudaError_t ce = cudaGetDeviceProperties(&prop, device);
    if (ce != cudaSuccess) { delete ctx; return fail(MAPF_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(ce)); }
    if (prop.major < 10) {
        delete ctx;
        return fail(MAPF_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major,
                    prop.minor);
    }
    const int sm_count = prop.multiProcessorCount;
    const size_t lut_bytes = (size_t)L * 5 * sizeof(u64);
    const size_t lut_pad = (lut_bytes + 15) & ~(size_t)15;
    sp.lut_bytes = (u32)lut_pad;
#define CTX_TRY(expr)                                                                                  \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess) {                                                                       \
            int _rc = fail(MAPF_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            mapf_ctx_destroy(ctx);                                                                     \
            return _rc;                                                                                \
        }                                                                                              \
    } while (0)
    const size_t image_head = MAPF_SMEM_LUT - MAPF_SMEM_IMG;  // pattern tables + action table
    CTX_TRY(cudaMalloc(&ctx->d_image, image_head + lut_pad));
    CTX_TRY(cudaMemset(ctx->d_image, 0, image_head + lut_pad));
    ctx->d_lut = reinterpret_cast<u64 *>(ctx->d_image + image_head);
    CTX_TRY(cudaMalloc(&ctx->d_cell_rc, (size_t)L * sizeof(u32)));
    CTX_TRY(cudaMalloc(&ctx->d_colbits, colbits.size() * sizeof(u32)));
    CTX_TRY(cudaMalloc(&ctx->d_colbase, colbase.size() * sizeof(u32)));
    CTX_TRY(cudaMemcpy(ctx->d_colbits, colbits.data(), colbits.size() * sizeof(u32), cudaMemcpyHostToDevice));
    CTX_TRY(cudaMemcpy(ctx->d_colbase, colbase.data(), colbase.size() * sizeof(u32), cudaMemcpyHostToDevice));
    {
        const size_t bm_smem = ((size_t)W * wpc + W) * sizeof(u32);
        if (bm_smem > (size_t)prop.sharedMemPerBlockOptin) {
            mapf_ctx_destroy(ctx);
            return fail(MAPF_ERR_UNSUPPORTED, "the %dx%d obstacle bitmap (%zu B) does not fit shared memory", H, W, bm_smem);
        }
        if (int rc = raise_smem_cap(device, (const void *)k_build_moves, bm_smem)) { mapf_ctx_destroy(ctx); return rc; }
        PatternList pats;
        memset(&pats, 0, sizeof(pats));
        pats.count = ctx->n_patterns;
        for (int p = 0; p < ctx->n_patterns; ++p) pats.triple[p] = ctx->pat_triple[p];
        const int blocks = (H * W + 255) / 256 < sm_count * 4 ? (H * W + 255) / 256 : sm_count * 4;
        GoalList goals;
        memset(&goals, 0, sizeof(goals));
        goals.n = n;
        for (int i = 0; i < n && i < 16; ++i) goals.cell[i] = (u16)goal_id[i];
        k_build_moves<<<blocks, 256, bm_smem>>>(ctx->d_colbits, ctx->d_colbase, H, W, wpc, sp.cand_mask, pats, goals,
                                                ctx->d_lut, ctx->d_cell_rc);
        CTX_TRY(cudaGetLastError());
        CTX_TRY(cudaDeviceSynchronize());
    }
    ctx->h_lut.resize((size_t)L * 5);
    ctx->h_cell_rc.resize(L);
    CTX_TRY(cudaMemcpy(ctx->h_lut.data(), ctx->d_lut, lut_bytes, cudaMemcpyDeviceToHost));
    CTX_TRY(cudaMemcpy(ctx->h_cell_rc.data(), ctx->d_cell_rc, (size_t)L * sizeof(u32), cudaMemcpyDeviceToHost));
    sp.lut = ctx->d_lut;

    // ---- launch geometry: stage the move table in shared memory when it leaves room for the per-warp scratch
    const size_t smem_limit = (size_t)prop.sharedMemPerBlockOptin;
    KernelSet probe;
    if (!pick_kernels(n, sp.words, true, &probe)) {
        mapf_ctx_destroy(ctx);
        return fail(MAPF_ERR_UNSUPPORTED, "no kernels for %d agents with %d-word states", n, sp.words);
    }
    ctx->threads = 512;  // two CTAs per SM stage the shared-memory image half as often as four of 256 (measured faster)
#ifdef MAPF_TUNING  // experiment builds only (make variant EXTRA=-DMAPF_TUNING): the release library reads no environment
    if (const char *e = getenv("MAPF_THREADS")) {
        const int t = atoi(e);
        if (t >= 32 && t <= MAPF_MAX_THREADS && t % 32 == 0) ctx->threads = t;
    }
#endif
    // (the shared-memory kernels also divide chunks on the fp64 pipe, which needs L**4 < 2**50 and L*L < 2**31)
    const bool luts = sp.divL.fix == 0 && (u128)sp.LL * sp.LL < ((u128)1 << 50) && sp.LL < (1u << 31) &&
                      MAPF_SMEM_LUT + lut_pad + (size_t)(ctx->threads / 32) * probe.backup_slab_bytes <= smem_limit;
    if (!luts) ctx->threads = 256;
    sp.lut_smem = luts ? 1 : 0;
    {
        // shared-window address of the hot kernels' dynamic shared memory (they have no static shared memory)
        u32 *d_probe = nullptr;
        CTX_TRY(cudaMalloc(&d_probe, sizeof(u32)));
        k_probe_smem<<<1, 32, 1024>>>(d_probe);
        CTX_TRY(cudaGetLastError());
        CTX_TRY(cudaMemcpy(&sp.smem_window, d_probe, sizeof(u32), cudaMemcpyDeviceToHost));
        cudaFree(d_probe);
        const u32 act0 = luts ? sp.smem_window + MAPF_SMEM_LUT : 0u;
        if (sp.smem_window & 0xffu) {  // ent_row() merges a pattern-row offset into the window address with one PRMT
            mapf_ctx_destroy(ctx);
            return fail(MAPF_ERR_UNSUPPORTED, "shared-memory window 0x%x is not a multiple of 256", sp.smem_window);
        }
        if (act0 + 32u > 0xffffu) {
            mapf_ctx_destroy(ctx);
            return fail(MAPF_ERR_UNSUPPORTED, "shared-memory window 0x%x does not fit the 16-bit action table", sp.smem_window);
        }
        std::vector<unsigned char> head(image_head, 0);
        memcpy(head.data() + (MAPF_SMEM_THR - MAPF_SMEM_IMG), ctx->pt.thr, sizeof(ctx->pt.thr));
        memcpy(head.data() + (MAPF_SMEM_CUM - MAPF_SMEM_IMG), ctx->pt.cum, sizeof(ctx->pt.cum));
        memcpy(head.data() + (MAPF_SMEM_PP - MAPF_SMEM_IMG), ctx->pt.pp, sizeof(ctx->pt.pp));
        memcpy(head.data() + (MAPF_SMEM_PZERO - MAPF_SMEM_IMG), ctx->pt.zero, sizeof(ctx->pt.zero));
        memcpy(head.data() + (MAPF_SMEM_REW - MAPF_SMEM_IMG), ctx->pt.reward, sizeof(ctx->pt.reward));
        uint16_t *act = reinterpret_cast<uint16_t *>(head.data() + (MAPF_SMEM_ACT - MAPF_SMEM_IMG));
        for (u32 a = 0; a < 625; ++a) {  // base-5 digits of a four-agent joint action (__init__.py:26, mapf_env.py:101-102)
            u32 x = a;
            for (int j = 0; j < 4; ++j) { act[a * 4 + j] = (uint16_t)(act0 + (x % 5u) * 8u); x /= 5u; }
        }
        CTX_TRY(cudaMemcpy(ctx->d_image, head.data(), image_head, cudaMemcpyHostToDevice));
        sp.image = ctx->d_image;
        sp.image_bytes = (u32)(image_head + (luts ? lut_pad : 0));
    }
    pick_kernels(n, sp.words, luts, &ctx->ks);
    ctx->smem_base = MAPF_SMEM_LUT + (luts ? lut_pad : 0);  // barrier + image
    ctx->threads_step = ctx->ks.step_threads ? ctx->ks.step_threads : ctx->threads;
    ctx->threads_expand = ctx->ks.expand_threads ? ctx->ks.expand_threads : ctx->threads;
    if (ctx->smem_base + (size_t)(ctx->threads_expand / 32) * ctx->ks.expand_slab_bytes > smem_limit)
        ctx->threads_expand = ctx->threads;  // the wide CTA's slabs do not fit next to this map's table
    ctx->smem_expand = ctx->smem_base + (size_t)(ctx->threads_expand / 32) * ctx->ks.expand_slab_bytes;
    ctx->smem_backup = ctx->smem_base + (size_t)(ctx->threads / 32) * ctx->ks.backup_slab_bytes;
    int grid_keep = 0;  // the KEEP kernels are launched with their plain twins' grids (host-link-bound callers)
    struct { const void *fn; size_t smem; int *grid; int threads; } plan[] = {
        {ctx->ks.step_philox1k, ctx->smem_base, &grid_keep, ctx->threads_step},
        {ctx->ks.step_philox2k, ctx->smem_base, &grid_keep},
        {ctx->ks.step_tape_k, ctx->smem_base, &grid_keep, ctx->threads_step},
        {ctx->ks.step_philox1ck, ctx->smem_base, &grid_keep, ctx->threads_step},
        {ctx->ks.step_philox2ck, ctx->smem_base, &grid_keep},
        {ctx->ks.step_tape_ck, ctx->smem_base, &grid_keep, ctx->threads_step},
        {ctx->ks.step_philox1, ctx->smem_base, &ctx->grid_step1, ctx->threads_step},
        {ctx->ks.step_philox2, ctx->smem_base, &ctx->grid_step2},
        {ctx->ks.step_tape, ctx->smem_base, &ctx->grid_step_tape, ctx->threads_step},
        {ctx->ks.step_philox1c, ctx->smem_base, &ctx->grid_step1, ctx->threads_step},
        {ctx->ks.step_philox2c, ctx->smem_base, &ctx->grid_step2},
        {ctx->ks.step_tape_c, ctx->smem_base, &ctx->grid_step_tape, ctx->threads_step},
        {ctx->ks.rollout_philox, ctx->smem_base, &ctx->grid_rollout},
        {ctx->ks.rollout_philox2, ctx->smem_base, &ctx->grid_rollout2, MAPF_ROLLOUT2_THREADS},
        {ctx->ks.rollout_philox2_rnd, ctx->smem_base, &ctx->grid_rollout2, MAPF_ROLLOUT2_THREADS},
        {ctx->ks.rollout_philox_rnd, ctx->smem_base, &ctx->grid_rollout},
        {ctx->ks.rollout_tape_rnd, ctx->smem_base, &ctx->grid_rollout_tape},
        {ctx->ks.rollout_tape, ctx->smem_base, &ctx->grid_rollout_tape},
        {ctx->ks.expand, ctx->smem_expand, &ctx->grid_expand, ctx->threads_expand},
        {ctx->ks.expand_range, ctx->smem_expand, &ctx->grid_expand_range, ctx->threads_expand},
        {ctx->ks.backup, ctx->smem_backup, &ctx->grid_backup},
        {ctx->ks.backup_range, ctx->smem_backup, &ctx->grid_backup_range},
        {ctx->ks.evaluate[MAPF_POLICY_RANDOM], ctx->smem_base, &ctx->grid_evaluate[MAPF_POLICY_RANDOM]},
        {ctx->ks.evaluate[MAPF_POLICY_JOINT], ctx->smem_base, &ctx->grid_evaluate[MAPF_POLICY_JOINT]},
        {ctx->ks.evaluate[MAPF_POLICY_AGENTS], ctx->smem_base, &ctx->grid_evaluate[MAPF_POLICY_AGENTS]},
        {ctx->ks.evaluate[MAPF_POLICY_GROUPS], ctx->smem_base, &ctx->grid_evaluate[MAPF_POLICY_GROUPS]},
        {ctx->ks.rtdp_backup, ctx->smem_backup, &ctx->grid_rtdp},
        {ctx->ks.evaluate_table, ctx->smem_base, &ctx->grid_evaluate_table}};
    for (auto &pl : plan) {
        if (!pl.fn) continue;  // two-word states have no backup kernels; wide step CTAs have no EPT = 2 k_step
        if (pl.smem > smem_limit) {
            mapf_ctx_destroy(ctx);
            return fail(MAPF_ERR_UNSUPPORTED, "a hot kernel needs %zu B of shared memory, the device offers %zu", pl.smem, smem_limit);
        }
        int rc = raise_smem_cap(device, pl.fn, pl.smem);
        if (!rc) rc = occupancy_grid(pl.fn, pl.threads ? pl.threads : ctx->threads, pl.smem, sm_count, pl.grid);
        if (rc) { mapf_ctx_destroy(ctx); return rc; }
#ifdef MAPF_TUNING
        if (const char *e = getenv("MAPF_BLOCKS_PER_SM")) {
            const int bps = atoi(e);
            if (bps >= 1 && bps * sm_count <= *pl.grid) *pl.grid = bps * sm_count;
        }
#endif
    }
    ctx->grid_plain = sm_count * 8;

    mapf_info &inf = ctx->info;
    memset(&inf, 0, sizeof(inf));
    inf.n_agents = n; inf.n_cells = L; inf.state_words = sp.words; inf.moves_in_smem = sp.lut_smem;
    inf.n_actions = (int64_t)nA;
    inf.n_states[0] = (u64)nS; inf.n_states[1] = (u64)(nS >> 64);
    inf.start_state[0] = (u64)s0; inf.start_state[1] = (u64)(s0 >> 64);
    inf.goal_state[0] = (u64)sg; inf.goal_state[1] = (u64)(sg >> 64);
    int64_t mr = 1;
    for (int i = 0; i < n; ++i) mr *= 3;
    inf.max_row_len = mr;
    inf.device = device; inf.sm_count = sm_count;
    *out = ctx;
    return MAPF_OK;
}

extern "C" int mapf_ctx_info(const mapf_ctx *ctx, mapf_info *out) {
    if (!ctx || !out) return fail(MAPF_ERR_INVALID, "mapf_ctx_info: NULL argument");
    *out = ctx->info;
    return MAPF_OK;
}

extern "C" int mapf_ctx_reward_table(const mapf_ctx *ctx, double out64[64]) {
    if (!ctx || !out64) return fail(MAPF_ERR_INVALID, "mapf_ctx_reward_table: NULL argument");
    static_assert(4 * MAPF_REW_STRIDE == 64, "reward table layout");
    memcpy(out64, ctx->pt.reward, 64 * sizeof(double));
    return MAPF_OK;
}

extern "C" int mapf_ctx_moves(const mapf_ctx *ctx, uint8_t *k, int32_t *dest, double *prob, int32_t *cells_rc) {
    if (!ctx) return fail(MAPF_ERR_INVALID, "mapf_ctx_moves: NULL context");
    const int L = ctx->sp.L;
    for (int i = 0; i < L * 5; ++i) {
        const u64 e = ctx->h_lut[i];
        const int kk = (int)ENT_K(e);
        const u32 pid = ENT_POFF(e) / MAPF_PAT_STRIDE;
        if (k) k[i] = (uint8_t)kk;
        for (int j = 0; j < 3; ++j) {
            if (dest) dest[i * 3 + j] = j < kk ? (int32_t)((e >> (16 * j)) & 0xffffu) : -1;
            if (prob) prob[i * 3 + j] = j < kk ? ctx->pt.pp[pid][j] : 0.0;
        }
    }
    if (cells_rc)
        for (int i = 0; i < L; ++i) {
            cells_rc[2 * i] = (int32_t)(ctx->h_cell_rc[i] >> 16);
            cells_rc[2 * i + 1] = (int32_t)(ctx->h_cell_rc[i] & 0xffffu);
        }
    return MAPF_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// launches
// ---------------------------------------------------------------------------------------------------------------
static int grid_for(int64_t work_items, int threads, int grid_max) {
    int64_t need = (work_items + threads - 1) / threads;
    if (need < 1) need = 1;
    return (int)(need < grid_max ? need : grid_max);
}

#define LAUNCH(fn, grid, threads, smem, stream, args)                                               \
    do {                                                                                            \
        cudaError_t _e = cudaLaunchKernel(fn, dim3(grid), dim3(threads), args, smem, (cudaStream_t)(stream)); \
        if (_e != cudaSuccess) return fail(MAPF_ERR_CUDA, "launch %s: %s", #fn, cudaGetErrorString(_e));      \
    } while (0)

// Two-word states are read and written as 16-byte vectors (load_state / store_state), so arrays of them must be
// 16-byte aligned: a misaligned one is rejected instead of faulting in the kernel.
static inline bool states_misaligned(int words, const void *p) { return words == 2 && ((uintptr_t)p & 15u) != 0; }

extern "C" int mapf_decode_states(const mapf_ctx *ctx, const void *states, int64_t B, int32_t *cells, void *stream) {
    if (!ctx || B < 0 || (B > 0 && (!states || !cells || states_misaligned(ctx->sp.words, states)))) return fail(MAPF_ERR_INVALID, "mapf_decode_states: bad argument");
    if (B == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    DevSpec sp = ctx->sp;
    void *args[] = {&sp, &states, &B, &cells};
    LAUNCH(ctx->ks.decode, grid_for(B, 256, ctx->grid_plain), 256, 0, stream, args);
    return MAPF_OK;
}

extern "C" int mapf_encode_states(const mapf_ctx *ctx, const int32_t *cells, int64_t B, void *states, void *stream) {
    if (!ctx || B < 0 || (B > 0 && (!states || !cells || states_misaligned(ctx->sp.words, states)))) return fail(MAPF_ERR_INVALID, "mapf_encode_states: bad argument");
    if (B == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    DevSpec sp = ctx->sp;
    void *args[] = {&sp, &cells, &B, &states};
    LAUNCH(ctx->ks.encode, grid_for(B, 256, ctx->grid_plain), 256, 0, stream, args);
    return MAPF_OK;
}

static int count_impl(const mapf_ctx *ctx, bool range, const void *states, const int32_t *actions, u64 sb_lo, u64 sb_hi,
                      int64_t B, int64_t *row_len, void *stream) {
    if (B == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    DevSpec sp = ctx->sp;
    void *args[] = {&sp, &states, &actions, &sb_lo, &sb_hi, &B, &row_len};
    LAUNCH(range ? ctx->ks.count_range : ctx->ks.count, grid_for(B, 256, ctx->grid_plain), 256, 0, stream, args);
    return MAPF_OK;
}

extern "C" int mapf_count_rows(const mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B,
                               int64_t *row_len, void *stream) {
    if (!ctx || B < 0 || (B > 0 && (!states || !actions || !row_len || states_misaligned(ctx->sp.words, states))))
        return fail(MAPF_ERR_INVALID, "mapf_count_rows: bad argument");
    return count_impl(ctx, false, states, actions, 0, 0, B, row_len, stream);
}

static int range_rows(const mapf_ctx *ctx, int64_t n_states, int64_t *B) {
    if (n_states < 0) return fail(MAPF_ERR_INVALID, "negative state count");
    if ((u128)n_states * (u128)ctx->sp.nA > (u128)0x7fffffffffffffffLL / 4)
        return fail(MAPF_ERR_INVALID, "slab of %lld states x %llu actions is too large for one call", (long long)n_states,
                    (unsigned long long)ctx->sp.nA);
    *B = n_states * (int64_t)ctx->sp.nA;
    return MAPF_OK;
}

extern "C" int mapf_count_range(const mapf_ctx *ctx, const uint64_t s_begin[2], int64_t n_states, int64_t *row_len,
                                void *stream) {
    if (!ctx || !s_begin || (n_states > 0 && !row_len)) return fail(MAPF_ERR_INVALID, "mapf_count_range: bad argument");
    int64_t B = 0;
    int rc = range_rows(ctx, n_states, &B);
    if (rc) return rc;
    return count_impl(ctx, true, nullptr, nullptr, s_begin[0], s_begin[1], B, row_len, stream);
}

// Launch behind the previous kernel of the stream with programmatic stream serialization: the grid may be scheduled while
// the predecessor drains (the kernel itself waits, grid_dependency_wait(), before it reads the predecessor's output).
template <typename... KArgs, typename... Args>
static cudaError_t launch_dependent(void (*kernel)(KArgs...), int grid, int threads, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(threads);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// count + scan in three launches instead of four (see k_count_partials)
static int count_scan_impl(const mapf_ctx *ctx, bool range, const void *states, const int32_t *actions, u64 sb_lo, u64 sb_hi,
                           int64_t B, int64_t *row_len, int64_t *row_ptr, void *scratch, void *stream) {
    if (!row_ptr || (B > 0 && !scratch)) return fail(MAPF_ERR_INVALID, "count_scan: NULL buffer");
    DeviceGuard g(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (B == 0) {
        CUDA_TRY(cudaMemsetAsync(row_ptr, 0, sizeof(int64_t), st));
        return MAPF_OK;
    }
    const int64_t chunks = (B + SCAN_CHUNK - 1) / SCAN_CHUNK;
    if (chunks > 0x7fffffff) return fail(MAPF_ERR_INVALID, "too many rows for one scan");
    DevSpec sp = ctx->sp;
    i64 *partial = (i64 *)scratch;
    const bool fold = chunks <= SCAN_FOLD_MAX_CHUNKS;  // every final block adds up the chunk totals before it itself
    const int nc = (int)chunks;
    if (row_len) {
        void *args[] = {&sp, &states, &actions, &sb_lo, &sb_hi, &B, &row_len, &partial};
        LAUNCH(range ? ctx->ks.count_partials_range : ctx->ks.count_partials, nc, 256, 0, stream, args);
        if (!fold) CUDA_TRY(launch_dependent(k_scan_spine, 1, SPINE_THREADS, st, partial, chunks));
        const int vec_ok = (((uintptr_t)row_len | (uintptr_t)row_ptr) & 15) == 0 ? 1 : 0;
        CUDA_TRY(launch_dependent(fold ? k_scan_final<true, i64> : k_scan_final<false, i64>, nc, 256, st, (const i64 *)row_len,
                                  B, (const i64 *)partial, (i64 *)row_ptr, vec_ok));
    } else {
        // the caller does not want the lengths: they live as u16 / u32 behind the chunk totals in the scratch
        // (mapf_scan_scratch_bytes reserves the room): 8 instead of 16 bytes per row travel between the two passes
        void *lens = (unsigned char *)scratch + (((size_t)(chunks + 1) * sizeof(i64) + 15) & ~(size_t)15);
        void *args[] = {&sp, &states, &actions, &sb_lo, &sb_hi, &B, &lens, &partial};
        LAUNCH(range ? ctx->ks.count_partials_range_c : ctx->ks.count_partials_c, nc, 256, 0, stream, args);
        if (!fold) CUDA_TRY(launch_dependent(k_scan_spine, 1, SPINE_THREADS, st, partial, chunks));
        const int vec_ok = ((uintptr_t)row_ptr & 15) == 0 ? 1 : 0;
        if (ctx->ks.compact_len_bytes == 2)
            CUDA_TRY(launch_dependent(fold ? k_scan_final<true, u16> : k_scan_final<false, u16>, nc, 256, st, (const u16 *)lens, B,
                                      (const i64 *)partial, (i64 *)row_ptr, vec_ok));
        else
            CUDA_TRY(launch_dependent(fold ? k_scan_final<true, u32> : k_scan_final<false, u32>, nc, 256, st, (const u32 *)lens, B,
                                      (const i64 *)partial, (i64 *)row_ptr, vec_ok));
    }
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

extern "C" int mapf_count_scan_rows(const mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B,
                                    int64_t *row_len, int64_t *row_ptr, void *scratch, void *stream) {
    if (!ctx || B < 0 || (B > 0 && (!states || !actions || states_misaligned(ctx->sp.words, states))))
        return fail(MAPF_ERR_INVALID, "mapf_count_scan_rows: bad argument");
    return count_scan_impl(ctx, false, states, actions, 0, 0, B, row_len, row_ptr, scratch, stream);
}

extern "C" int mapf_count_scan_range(const mapf_ctx *ctx, const uint64_t s_begin[2], int64_t n_states, int64_t *row_len,
                                     int64_t *row_ptr, void *scratch, void *stream) {
    if (!ctx || !s_begin) return fail(MAPF_ERR_INVALID, "mapf_count_scan_range: bad argument");
    int64_t B = 0;
    int rc = range_rows(ctx, n_states, &B);
    if (rc) return rc;
    return count_scan_impl(ctx, true, nullptr, nullptr, s_begin[0], s_begin[1], B, row_len, row_ptr, scratch, stream);
}

extern "C" int64_t mapf_scan_scratch_bytes(int64_t B) {
    int64_t chunks = (B + SCAN_CHUNK - 1) / SCAN_CHUNK;
    if (chunks < 1) chunks = 1;
    // chunk totals + (16-byte aligned) room for compact u32 row lengths, used when mapf_count_scan_* gets row_len = NULL
    return (((chunks + 1) * (int64_t)sizeof(int64_t) + 15) & ~(int64_t)15) + (B < 0 ? 0 : B) * 4 + 16;
}

extern "C" int mapf_scan_rows(const mapf_ctx *ctx, const int64_t *row_len, int64_t B, int64_t *row_ptr, void *scratch,
                              void *stream) {
    if (!ctx || B < 0 || !row_ptr || (B > 0 && (!row_len || !scratch)))
        return fail(MAPF_ERR_INVALID, "mapf_scan_rows: bad argument");
    DeviceGuard g(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (B == 0) {
        CUDA_TRY(cudaMemsetAsync(row_ptr, 0, sizeof(int64_t), st));
        return MAPF_OK;
    }
    const int64_t chunks = (B + SCAN_CHUNK - 1) / SCAN_CHUNK;
    if (chunks > 0x7fffffff) return fail(MAPF_ERR_INVALID, "too many rows for one scan");
    i64 *partial = (i64 *)scratch;
    k_scan_partials<<<(int)chunks, 256, 0, st>>>((const i64 *)row_len, B, partial);
    const int vec_ok = (((uintptr_t)row_len | (uintptr_t)row_ptr) & 15) == 0 ? 1 : 0;
    const bool fold = chunks <= SCAN_FOLD_MAX_CHUNKS;
    if (!fold) CUDA_TRY(launch_dependent(k_scan_spine, 1, SPINE_THREADS, st, partial, chunks));
    CUDA_TRY(launch_dependent(fold ? k_scan_final<true, i64> : k_scan_final<false, i64>, (int)chunks, 256, st,
                              (const i64 *)row_len, B, (const i64 *)partial, (i64 *)row_ptr, vec_ok));
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

static int expand_impl(const mapf_ctx *ctx, bool range, const void *states, const int32_t *actions, u64 sb_lo, u64 sb_hi,
                       int64_t B, const int64_t *row_ptr, void *next_state, double *prob, double *reward, uint8_t *flags,
                       void *stream) {
    if (B == 0) return MAPF_OK;
    if (!row_ptr || !next_state || !prob || !reward || !flags) return fail(MAPF_ERR_INVALID, "expand: NULL output");
    DeviceGuard g(ctx->device);
    DevSpec sp = ctx->sp;
    void *args[] = {&sp, &states, &actions, &sb_lo, &sb_hi, &B, &row_ptr, &next_state, &prob, &reward, &flags};
    // Work is cut by records (at least 32 per warp); their number is only known on the device, B * 3**n bounds it.
    const double rec_max = (double)B * (double)ctx->info.max_row_len;
    const int64_t lanes = rec_max > 4e18 ? (int64_t)4e18 : (int64_t)rec_max;
    const int grid = grid_for(lanes, ctx->threads_expand, range ? ctx->grid_expand_range : ctx->grid_expand);
    LAUNCH(range ? ctx->ks.expand_range : ctx->ks.expand, grid, ctx->threads_expand, ctx->smem_expand, stream, args);
    return MAPF_OK;
}

extern "C" int mapf_expand(const mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B,
                           const int64_t *row_ptr, void *next_state, double *prob, double *reward, uint8_t *flags,
                           void *stream) {
    if (!ctx || B < 0 || (B > 0 && (!states || !actions || states_misaligned(ctx->sp.words, states) ||
                                     states_misaligned(ctx->sp.words, next_state))))
        return fail(MAPF_ERR_INVALID, "mapf_expand: bad argument");
    return expand_impl(ctx, false, states, actions, 0, 0, B, row_ptr, next_state, prob, reward, flags, stream);
}

extern "C" int mapf_expand_range(const mapf_ctx *ctx, const uint64_t s_begin[2], int64_t n_states, const int64_t *row_ptr,
                                 void *next_state, double *prob, double *reward, uint8_t *flags, void *stream) {
    if (!ctx || !s_begin) return fail(MAPF_ERR_INVALID, "mapf_expand_range: bad argument");
    int64_t B = 0;
    int rc = range_rows(ctx, n_states, &B);
    if (rc) return rc;
    return expand_impl(ctx, true, nullptr, nullptr, s_begin[0], s_begin[1], B, row_ptr, next_state, prob, reward, flags,
                       stream);
}

extern "C" int mapf_checksum(const mapf_ctx *ctx, int64_t n_records, int64_t index_base, const void *next_state,
                             const double *prob, const double *reward, const uint8_t *flags, uint64_t *out8, void *stream) {
    if (!ctx || n_records < 0 || !out8 ||
        (n_records > 0 && (!next_state || !prob || !reward || !flags || states_misaligned(ctx->sp.words, next_state))))
        return fail(MAPF_ERR_INVALID, "mapf_checksum: bad argument");
    if (n_records == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    k_checksum<<<grid_for(n_records, 256, ctx->grid_plain), 256, 0, (cudaStream_t)stream>>>(
        ctx->sp.words, n_records, index_base, (const u64 *)next_state, prob, reward, flags, (u64 *)out8);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// rows next to the hot path: Bellman backup, predecessors, local-view projection
// ---------------------------------------------------------------------------------------------------------------
static int backup_impl(const mapf_ctx *ctx, bool range, const void *states, const int32_t *actions, u64 sb_lo, int64_t B,
                       const double *V, int64_t v_len, double gamma, double *Q, void *stream) {
    if (ctx->sp.words != 1)
        return fail(MAPF_ERR_UNSUPPORTED, "backup: a value vector over L**n = %d**%d states cannot exist", ctx->sp.L, ctx->sp.n);
    if (!V || !Q || v_len < 0 || (u64)v_len <= ctx->sp.smax[0])
        return fail(MAPF_ERR_INVALID, "backup: V must hold nS = %llu values (v_len = %lld)",
                    (unsigned long long)ctx->sp.smax[0] + 1, (long long)v_len);
    if (B == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    DevSpec sp = ctx->sp;
    void *args[] = {&sp, &states, &actions, &sb_lo, &B, &V, &gamma, &Q};
    const int grid = grid_for(B, ctx->threads, range ? ctx->grid_backup_range : ctx->grid_backup);
    LAUNCH(range ? ctx->ks.backup_range : ctx->ks.backup, grid, ctx->threads, ctx->smem_backup, stream, args);
    return MAPF_OK;
}

extern "C" int mapf_backup(const mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B, const double *V,
                           int64_t v_len, double gamma, double *Q, void *stream) {
    if (!ctx || B < 0 || (B > 0 && (!states || !actions))) return fail(MAPF_ERR_INVALID, "mapf_backup: bad argument");
    return backup_impl(ctx, false, states, actions, 0, B, V, v_len, gamma, Q, stream);
}

extern "C" int mapf_backup_range(const mapf_ctx *ctx, const uint64_t s_begin[2], int64_t n_states, const double *V,
                                 int64_t v_len, double gamma, double *Q, void *stream) {
    if (!ctx || !s_begin) return fail(MAPF_ERR_INVALID, "mapf_backup_range: bad argument");
    int64_t B = 0;
    int rc = range_rows(ctx, n_states, &B);
    if (rc) return rc;
    if (s_begin[1] != 0 || (n_states > 0 && s_begin[0] + (u64)n_states - 1 > ctx->sp.smax[0]))
        return fail(MAPF_ERR_INVALID, "mapf_backup_range: the slab leaves the state space");
    return backup_impl(ctx, true, nullptr, nullptr, s_begin[0], B, V, v_len, gamma, Q, stream);
}

static int greedy_impl(const mapf_ctx *ctx, const double *Q, int64_t n_states, double *V_out, int32_t *policy,
                       const PeerList &peers, int64_t s_begin, void *stream) {
    if (n_states == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    const int64_t nA = (int64_t)ctx->sp.nA;
    k_greedy<<<grid_for(((n_states + 31) / 32) * 32, 256, ctx->grid_plain), 256, 0, (cudaStream_t)stream>>>(
        Q, n_states, nA, V_out, policy, peers, s_begin);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

extern "C" int mapf_greedy(const mapf_ctx *ctx, const double *Q, int64_t n_states, double *V_out, int32_t *policy,
                           void *stream) {
    if (!ctx || n_states < 0 || (n_states > 0 && !Q)) return fail(MAPF_ERR_INVALID, "mapf_greedy: bad argument");
    PeerList none;
    memset(&none, 0, sizeof(none));
    return greedy_impl(ctx, Q, n_states, V_out, policy, none, 0, stream);
}

extern "C" int mapf_greedy_bcast(const mapf_ctx *ctx, const double *Q, int64_t n_states, int64_t s_begin,
                                 double *const *peer_values, int32_t n_peers, int32_t *policy, void *stream) {
    if (!ctx || n_states < 0 || s_begin < 0 || !peer_values || n_peers < 1 || n_peers > 16 || (n_states > 0 && !Q))
        return fail(MAPF_ERR_INVALID, "mapf_greedy_bcast: bad argument (1..16 peers)");
    PeerList peers;
    memset(&peers, 0, sizeof(peers));
    peers.n = n_peers;
    for (int r = 0; r < n_peers; ++r) {
        if (!peer_values[r]) return fail(MAPF_ERR_INVALID, "mapf_greedy_bcast: NULL peer pointer %d", r);
        peers.ptr[r] = peer_values[r];
    }
    return greedy_impl(ctx, Q, n_states, nullptr, policy, peers, s_begin, stream);
}

extern "C" int mapf_count_predecessors(const mapf_ctx *ctx, const void *states, int64_t B, int64_t *row_len, void *stream) {
    if (!ctx || B < 0 || (B > 0 && (!states || !row_len || states_misaligned(ctx->sp.words, states))))
        return fail(MAPF_ERR_INVALID, "mapf_count_predecessors: bad argument");
    if (B == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    DevSpec sp = ctx->sp;
    void *args[] = {&sp, &states, &B, &row_len};
    LAUNCH(ctx->ks.pred_count, grid_for(B, 256, ctx->grid_plain), 256, 0, stream, args);
    return MAPF_OK;
}

extern "C" int mapf_predecessors(const mapf_ctx *ctx, const void *states, int64_t B, const int64_t *row_ptr, void *pred,
                                 void *stream) {
    if (!ctx || B < 0 || (B > 0 && (!states || !row_ptr || !pred || states_misaligned(ctx->sp.words, states) ||
                                     states_misaligned(ctx->sp.words, pred))))
        return fail(MAPF_ERR_INVALID, "mapf_predecessors: bad argument");
    if (B == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    DevSpec sp = ctx->sp;
    void *args[] = {&sp, &states, &B, &row_ptr, &pred};
    LAUNCH(ctx->ks.pred_emit, grid_for(B * 32, 256, ctx->grid_plain), 256, 0, stream, args);
    return MAPF_OK;
}

extern "C" int mapf_projected_words(const mapf_ctx *ctx, int32_t n_sub) {
    if (!ctx || n_sub < 1 || n_sub > ctx->sp.n) return fail(MAPF_ERR_INVALID, "mapf_projected_words: bad argument");
    u128 v = 1;
    for (int i = 0; i < n_sub; ++i) v *= (u128)ctx->sp.L;
    return v < ((u128)1 << 63) ? 1 : 2;
}

extern "C" int mapf_project_states(const mapf_ctx *ctx, const void *states, int64_t B, const int32_t *agents, int32_t n_sub,
                                   void *out_states, void *stream) {
    if (!ctx || B < 0 || !agents || n_sub < 1 || n_sub > ctx->sp.n ||
        (B > 0 && (!states || !out_states || states_misaligned(ctx->sp.words, states) ||
                   states_misaligned(mapf_projected_words(ctx, n_sub), out_states))))
        return fail(MAPF_ERR_INVALID, "mapf_project_states: bad argument");
    AgentList sub;
    memset(&sub, 0, sizeof(sub));
    sub.n = n_sub;
    for (int j = 0; j < n_sub; ++j) {
        if (agents[j] < 0 || agents[j] >= ctx->sp.n) return fail(MAPF_ERR_INVALID, "agent index %d out of range", agents[j]);
        for (int q = 0; q < j; ++q)
            if (agents[q] == agents[j]) return fail(MAPF_ERR_INVALID, "agent index %d listed twice", agents[j]);
        sub.idx[j] = agents[j];
    }
    sub.words_out = mapf_projected_words(ctx, n_sub);
    if (B == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    DevSpec sp = ctx->sp;
    void *args[] = {&sp, &states, &B, &sub, &out_states};
    LAUNCH(ctx->ks.project, grid_for(B, 256, ctx->grid_plain), 256, 0, stream, args);
    return MAPF_OK;
}

static inline bool aligned(const void *p, size_t a) { return ((uintptr_t)p & (a - 1)) == 0; }

static PhiloxKeys make_keys(uint64_t seed) {
    PhiloxKeys K;
    u32 k0 = (u32)seed, k1 = (u32)(seed >> 32);
    for (int r = 0; r < 10; ++r) {
        K.k[2 * r] = k0;
        K.k[2 * r + 1] = k1;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return K;
}

#define MAPF_SMALL_HOST_BATCH 1024         // mapf_step_host: batches up to this size go through the pinned scratch
#define MAPF_LAUNCH_MAX_ENVS (1ll << 30)  // kernels index envs with 32 bits; larger batches are split

// CTA size of a grid-stride k_step launch over `items` work items (envs / EPT) on at most `*grid` CTAs of at most
// `max_threads` threads, for a kernel of which `per_sm` CTAs are resident on an SM.  The items need
// rounds = ceil(items / (grid * max_threads)) grid-stride rounds; the CTA is then the smallest size that covers the items
// in that many rounds, so that all threads run the same number of rounds, give or take one, and no part of the grid
// idles through a last round that only some CTAs have.  Example: one pool of 2**19 C2 envs (2**18 pairs) on 148 CTAs:
// 512 threads run 3.46 rounds each (68 CTAs run a 4th, 80 sit it out), 448 threads run 3.95.  The size is a multiple of
// 4 / gcd(per_sm, 4) warps, so that the resident warps of an SM split evenly over its four schedulers (measured on
// 2**20 C2 envs: 416 and 480 threads, 26 and 30 warps per SM, are 10 % slower than 448 and 512).  The grid shrinks only
// where CTAs would get no item.  A smaller CTA is always legal under the kernel's __launch_bounds__ and keeps the
// occupancy the grid was sized for; results depend on the env index only.
static int plan_step_cta(u32 items, int max_threads, int per_sm, int *grid) {
    const int quantum = 32 * (per_sm % 4 == 0 ? 1 : per_sm % 2 == 0 ? 2 : 4);
    const int64_t g = *grid, rounds = ((int64_t)items + g * max_threads - 1) / (g * max_threads);
    int threads = (int)(((int64_t)items + g * rounds * quantum - 1) / (g * rounds * quantum)) * quantum;
    if (threads > max_threads) threads = max_threads;  // a max_threads that is not a multiple of the quantum
    const int64_t used = ((int64_t)items + threads - 1) / threads;
    if (used < g) *grid = (int)used;
    return threads;
}

// Picks the step-kernel variant: replayed uniforms -> TAPE; otherwise the 2-envs-per-thread kernel with 128-bit
// loads/stores when the batch is even and every buffer is suitably aligned, else the scalar one.
static int launch_step(const mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B, const double *uniforms,
                       uint64_t seed, uint64_t step_index, int64_t env_offset, uint32_t options, void *next_states,
                       double *reward, double *prob, uint8_t *done, uint8_t *collision, cudaStream_t stream,
                       int grid_limit = 0, void *keep = nullptr) {
    if (!uniforms && !ctx->philox_ok)
        return fail(MAPF_ERR_UNSUPPORTED, "device-side sampling needs slip probabilities that add up to 1; pass uniforms");
    const size_t sw = (size_t)ctx->sp.words * 8;
#ifdef MAPF_TUNING
    static int force_ept = -1;
    if (force_ept < 0) {
        const char *e = getenv("MAPF_STEP_EPT");
        force_ept = e ? atoi(e) : 0;
    }
#else
    constexpr int force_ept = 0;
#endif
    for (int64_t off = 0; off < B; off += MAPF_LAUNCH_MAX_ENVS) {
        const int64_t nb64 = B - off < MAPF_LAUNCH_MAX_ENVS ? B - off : MAPF_LAUNCH_MAX_ENVS;
        DevSpec sp = ctx->sp;
        PhiloxKeys keys = make_keys(seed);
        const void *a_states = (const unsigned char *)states + sw * off;
        const int32_t *a_actions = actions + off;
        const double *a_u = uniforms ? uniforms + (size_t)off * ctx->sp.n : nullptr;
        void *a_ns = (unsigned char *)next_states + sw * off;
        const bool compact = (options & MAPF_OPT_COMPACT) != 0;  // reward codes are one byte per env
        double *a_r = compact ? (double *)((uint8_t *)reward + off) : reward + off, *a_p = prob + off;
        uint8_t *a_d = done + off, *a_c = collision ? collision + off : nullptr;
        void *a_keep = keep ? (unsigned char *)keep + sw * off : nullptr;  // KEEP kernels: second copy of the next states
        u32 nb = (u32)nb64;
        u64 st = step_index, e0 = (u64)(env_offset + off);
        u32 op = options;
#ifdef MAPF_TRACE  // timeline builds: the Philox-mode kernel receives the trace buffer in place of the unused uniforms
        const double *trace_buf = nullptr;
        if (!uniforms) {
            if (const char *e = getenv("MAPF_TRACE_PTR")) trace_buf = (const double *)strtoull(e, nullptr, 0);
        }
        void *args[] = {&sp, &keys, &a_states, &a_actions, &nb, uniforms ? (void *)&a_u : (void *)&trace_buf, &st, &e0, &op,
                        &a_ns, &a_r, &a_p, &a_d, &a_c, &a_keep};
#else
        void *args[] = {&sp, &keys, &a_states, &a_actions, &nb, &a_u, &st, &e0, &op, &a_ns, &a_r, &a_p, &a_d, &a_c, &a_keep};
#endif
        const void *fn;
        int grid;
        const KernelSet &ks = ctx->ks;
        int max_threads = ctx->threads;
        u32 items = nb;  // grid-stride work items: envs / EPT
        if (uniforms) {
            fn = keep ? (compact ? ks.step_tape_ck : ks.step_tape_k) : (compact ? ks.step_tape_c : ks.step_tape);
            max_threads = ctx->threads_step;
            grid = ctx->grid_step_tape;
        } else if (force_ept != 1 && ks.step_philox2 && (nb & 1) == 0 && aligned(a_states, 16) && aligned(a_ns, 16) && aligned(a_actions, 8) &&
                   aligned(a_r, compact ? 2 : 16) && aligned(a_p, 16) && aligned(a_d, 2) && (compact || aligned(a_c, 2)) &&
                   aligned(a_keep, 16)) {
            fn = keep ? (compact ? ks.step_philox2ck : ks.step_philox2k) : (compact ? ks.step_philox2c : ks.step_philox2);
            grid = ctx->grid_step2;
            items = nb / 2;
        } else {
            fn = keep ? (compact ? ks.step_philox1ck : ks.step_philox1k) : (compact ? ks.step_philox1c : ks.step_philox1);
            max_threads = ctx->threads_step;
            grid = ctx->grid_step1;
        }
        const int per_sm = grid / ctx->info.sm_count;  // the grids above are the kernels' resident CTAs on every SM
        if (grid_limit > 0 && grid > grid_limit) grid = grid_limit;
        if ((options & MAPF_OPT_SHARE_SM) && grid > ctx->info.sm_count) grid = ctx->info.sm_count;
        // Only the pools' launches (one CTA per SM each) are sized by plan_step_cta: two pools of 2**19 C2 envs step in
        // 8.89 us instead of 9.18 with 448-thread CTAs, while a single chain of 2**20 envs (two CTAs of one launch per SM)
        // runs 1.0 % slower at 448 threads than at 512 (profiles/r04_launch_shape.txt).
        int threads = max_threads;
        if (options & MAPF_OPT_SHARE_SM) threads = plan_step_cta(items, max_threads, per_sm, &grid);
        else grid = grid_for(items, threads, grid);
#ifdef MAPF_TUNING
        static int use_pdl = -1;
        if (use_pdl < 0) {
            const char *e = getenv("MAPF_PDL");
            use_pdl = e ? atoi(e) : 1;
        }
#else
        constexpr int use_pdl = 1;
#endif
        if (use_pdl) {
            // programmatic stream serialization: this launch may begin (up to its griddepcontrol.wait) while the
            // previous kernel of the stream is still draining
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(grid);
            cfg.blockDim = dim3(threads);
            cfg.dynamicSmemBytes = ctx->smem_base;
            cfg.stream = stream;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            cudaError_t e = cudaLaunchKernelExC(&cfg, fn, args);
            if (e != cudaSuccess) return fail(MAPF_ERR_CUDA, "launch k_step: %s", cudaGetErrorString(e));
        } else {
            LAUNCH(fn, grid, threads, ctx->smem_base, stream, args);
        }
    }
    return MAPF_OK;
}

extern "C" int mapf_step(const mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B,
                         const double *uniforms, uint64_t seed, uint64_t step_index, int64_t env_offset,
                         uint32_t options, void *next_states, double *reward, double *prob, uint8_t *done,
                         uint8_t *collision, void *stream) {
    if (!ctx || B < 0 || (B > 0 && (!states || !actions || !next_states || !reward || !prob || !done ||
                                     (!collision && !(options & MAPF_OPT_COMPACT)) ||
                                     states_misaligned(ctx->sp.words, states) || states_misaligned(ctx->sp.words, next_states))))
        return fail(MAPF_ERR_INVALID, "mapf_step: bad argument");
    if (B == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    return launch_step(ctx, states, actions, B, uniforms, seed, step_index, env_offset, options, next_states, reward, prob,
                       done, collision, (cudaStream_t)stream);
}

extern "C" int mapf_rollout(const mapf_ctx *ctx, void *states_inout, const int32_t *actions, int64_t T, int64_t B,
                            const double *uniforms, uint64_t seed, uint64_t step_index0, int64_t env_offset,
                            uint32_t options, void *next_states, double *reward, double *prob, uint8_t *done,
                            uint8_t *collision, void *stream) {
    if (!ctx || B < 0 || T < 0 ||
        (B > 0 && T > 0 && (!states_inout || !next_states || !reward || !prob || !done || !collision ||
                            states_misaligned(ctx->sp.words, states_inout) || states_misaligned(ctx->sp.words, next_states))))
        return fail(MAPF_ERR_INVALID, "mapf_rollout: bad argument");
    if (B == 0 || T == 0) return MAPF_OK;
    if (B > MAPF_LAUNCH_MAX_ENVS) return fail(MAPF_ERR_INVALID, "mapf_rollout: at most 2**30 envs per call");
    if (!uniforms && !ctx->philox_ok)
        return fail(MAPF_ERR_UNSUPPORTED, "device-side sampling needs slip probabilities that add up to 1; pass uniforms");
    DeviceGuard g(ctx->device);
    DevSpec sp = ctx->sp;
    PhiloxKeys keys = make_keys(seed);
    u64 st = step_index0, e0 = (u64)env_offset;
    u32 op = options, nb = (u32)B;
    void *args[] = {&sp, &keys, &states_inout, &actions, &T, &nb, &uniforms, &st, &e0, &op, &next_states, &reward, &prob,
                    &done, &collision};
    const bool given = actions != nullptr;
    if (uniforms) {
        LAUNCH(given ? ctx->ks.rollout_tape : ctx->ks.rollout_tape_rnd, grid_for(B, ctx->threads, ctx->grid_rollout_tape),
               ctx->threads, ctx->smem_base, stream, args);
    } else if (ctx->ks.rollout_philox2 && (B & 1) == 0 && aligned(states_inout, 16) && aligned(next_states, 16) &&
               (!actions || aligned(actions, 8)) && aligned(reward, 16) && aligned(prob, 16) && aligned(done, 2) &&
               aligned(collision, 2)) {
        // two envs per thread, 128-bit stores: every slab t * B of the [T, B] outputs keeps the base alignment (B even)
        LAUNCH(given ? ctx->ks.rollout_philox2 : ctx->ks.rollout_philox2_rnd,
               grid_for(B / 2, MAPF_ROLLOUT2_THREADS, ctx->grid_rollout2), MAPF_ROLLOUT2_THREADS, ctx->smem_base, stream, args);
    } else {
        LAUNCH(given ? ctx->ks.rollout_philox : ctx->ks.rollout_philox_rnd, grid_for(B, ctx->threads, ctx->grid_rollout),
               ctx->threads, ctx->smem_base, stream, args);
    }
    return MAPF_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// closed-loop policy evaluation
// ---------------------------------------------------------------------------------------------------------------
extern "C" int64_t mapf_evaluate_scratch_bytes(void) { return 16; }  // the u32 episode queue counter, padded

extern "C" int mapf_evaluate(const mapf_ctx *ctx, int32_t policy_kind, const void *policy, int64_t policy_len,
                             int64_t n_episodes, int64_t max_steps, double gamma, uint64_t seed, uint64_t step_index0,
                             int64_t episode_offset, void *scratch, double *ret, int32_t *length, uint8_t *outcome,
                             void *stream) {
    if (!ctx || policy_kind < MAPF_POLICY_RANDOM || policy_kind > MAPF_POLICY_AGENTS || n_episodes < 0 ||
        (policy_kind != MAPF_POLICY_RANDOM && !policy) || (n_episodes > 0 && (!scratch || !ret || !length || !outcome)))
        return fail(MAPF_ERR_INVALID, "mapf_evaluate: bad argument");
    if (max_steps < 1 || max_steps >= (1ll << 31))
        return fail(MAPF_ERR_INVALID, "mapf_evaluate: max_steps = %lld, must be in [1, 2**31)", (long long)max_steps);
    if (n_episodes > MAPF_LAUNCH_MAX_ENVS) return fail(MAPF_ERR_INVALID, "mapf_evaluate: at most 2**30 episodes per call");
    if (policy_kind == MAPF_POLICY_JOINT) {
        if (ctx->sp.words != 1)
            return fail(MAPF_ERR_UNSUPPORTED, "mapf_evaluate: a joint-state policy over L**n = %d**%d states cannot exist; "
                                              "use MAPF_POLICY_AGENTS", ctx->sp.L, ctx->sp.n);
        if (policy_len < 0 || (u64)policy_len <= ctx->sp.smax[0])
            return fail(MAPF_ERR_INVALID, "mapf_evaluate: a joint-state policy needs nS = %llu entries (policy_len = %lld)",
                        (unsigned long long)ctx->sp.smax[0] + 1, (long long)policy_len);
    }
    if (policy_kind == MAPF_POLICY_AGENTS && policy_len != (int64_t)ctx->sp.n * ctx->sp.L)
        return fail(MAPF_ERR_INVALID, "mapf_evaluate: a per-agent policy has n * L = %lld entries (policy_len = %lld)",
                    (long long)ctx->sp.n * ctx->sp.L, (long long)policy_len);
    if (!ctx->philox_ok)
        return fail(MAPF_ERR_UNSUPPORTED, "device-side sampling needs slip probabilities that add up to 1");
    if (n_episodes == 0) return MAPF_OK;
    const void *fn = ctx->ks.evaluate[policy_kind];
    if (!fn) return fail(MAPF_ERR_UNSUPPORTED, "mapf_evaluate: no kernel for policy kind %d", policy_kind);
    DeviceGuard g(ctx->device);
    CUDA_TRY(cudaMemsetAsync(scratch, 0, sizeof(u32), (cudaStream_t)stream));
    DevSpec sp = ctx->sp;
    PhiloxKeys keys = make_keys(seed);
    u32 E = (u32)n_episodes, T = (u32)max_steps;
    u64 st = step_index0, e0 = (u64)episode_offset;
    void *args[] = {&sp, &keys, &policy, &E, &T, &gamma, &st, &e0, &scratch, &ret, &length, &outcome};
    LAUNCH(fn, grid_for(n_episodes, ctx->threads, ctx->grid_evaluate[policy_kind]), ctx->threads, ctx->smem_base, stream,
           args);
    return MAPF_OK;
}

// The agent groups of a group_of / table-length pair (mapf_evaluate_groups' rules), as the per-agent GroupLayout of the
// kernels; *heads gets bit i set when agent i is the first agent of its group.  `who` names the entry point in errors.
static int group_layout(const mapf_ctx *ctx, const char *who, const int32_t *group_of, int64_t tables_len, GroupLayout *gl,
                        u32 *heads) {
    const int n = ctx->sp.n;
    const u64 L = (u64)ctx->sp.L;
    int size[MAPF_MAXN] = {0}, pos[MAPF_MAXN], n_groups = 0;
    for (int i = 0; i < n; ++i) {
        const int g = group_of[i];
        if (g < 0 || g > n_groups)  // canonical: a new group takes the next id
            return fail(MAPF_ERR_INVALID, "%s: group_of[%d] = %d, must be in [0, %d]", who, i, g, n_groups);
        if (g == n_groups) ++n_groups;
        pos[i] = size[g]++;
    }
    // table g holds L**size[g] entries at first[g]; every partial sum stays below 2**63
    u64 first[MAPF_MAXN], total = 0, powL[MAPF_MAXN + 1];
    powL[0] = 1;
    for (int k = 1; k <= n; ++k) powL[k] = powL[k - 1] > (u64)INT64_MAX / L ? (u64)INT64_MAX : powL[k - 1] * L;
    for (int g = 0; g < n_groups; ++g) {
        if (powL[size[g]] == (u64)INT64_MAX || total > (u64)INT64_MAX - powL[size[g]])
            return fail(MAPF_ERR_INVALID, "%s: the tables have more than 2**63 - 1 entries", who);
        first[g] = total;
        total += powL[size[g]];
    }
    if (tables_len < 0 || (u64)tables_len != total)
        return fail(MAPF_ERR_INVALID, "%s: the groups' tables have %llu entries (tables_len = %lld)", who,
                    (unsigned long long)total, (long long)tables_len);
    memset(gl, 0, sizeof(*gl));
    *heads = 0;
    for (int i = 0; i < n; ++i) {
        const int g = group_of[i];
        for (int j = 0; j < n; ++j) gl->mul[i][j] = group_of[j] == g ? powL[pos[j]] : 0;
        gl->off[i] = first[g];
        u64 d = 5;  // 5**(pos[i] + 1) <= 5**13 < 2**32: not a divisor of 2**64, so the ceiling is floor + 1
        for (int k = 0; k < pos[i]; ++k) d *= 5;
        gl->frac[i] = ~0ull / d + 1;
        u32 a = 1;
        for (int k = 0; k < size[g]; ++k) a *= 5u;
        gl->amax[i] = a - 1u;
        gl->group[i] = (u32)g;
        if (pos[i] == 0) *heads |= 1u << i;
    }
    return MAPF_OK;
}

extern "C" int mapf_evaluate_groups(const mapf_ctx *ctx, const int32_t *group_of, const int32_t *tables,
                                    int64_t tables_len, int64_t n_episodes, int64_t max_steps, double gamma,
                                    uint64_t seed, uint64_t step_index0, int64_t episode_offset, void *scratch,
                                    double *ret, int32_t *length, uint8_t *outcome, uint8_t *conflict, void *stream) {
    if (!ctx || !group_of || !tables || n_episodes < 0 || (n_episodes > 0 && (!scratch || !ret || !length || !outcome)))
        return fail(MAPF_ERR_INVALID, "mapf_evaluate_groups: bad argument");
    if (max_steps < 1 || max_steps >= (1ll << 31))
        return fail(MAPF_ERR_INVALID, "mapf_evaluate_groups: max_steps = %lld, must be in [1, 2**31)", (long long)max_steps);
    if (n_episodes > MAPF_LAUNCH_MAX_ENVS)
        return fail(MAPF_ERR_INVALID, "mapf_evaluate_groups: at most 2**30 episodes per call");
    GroupLayout gl;
    u32 heads;
    const int rc = group_layout(ctx, "mapf_evaluate_groups", group_of, tables_len, &gl, &heads);
    if (rc) return rc;
    if (!ctx->philox_ok)
        return fail(MAPF_ERR_UNSUPPORTED, "device-side sampling needs slip probabilities that add up to 1");
    if (n_episodes == 0) return MAPF_OK;
    const void *fn = ctx->ks.evaluate[MAPF_POLICY_GROUPS];
    if (!fn) return fail(MAPF_ERR_UNSUPPORTED, "mapf_evaluate_groups: no kernel");
    DeviceGuard dg(ctx->device);
    CUDA_TRY(cudaMemsetAsync(scratch, 0, sizeof(u32), (cudaStream_t)stream));
    DevSpec sp = ctx->sp;
    PhiloxKeys keys = make_keys(seed);
    u32 E = (u32)n_episodes, T = (u32)max_steps;
    u64 st = step_index0, e0 = (u64)episode_offset;
    void *args[] = {&sp, &keys, &tables, &gl, &E, &T, &gamma, &st, &e0, &scratch, &ret, &length, &outcome, &conflict};
    LAUNCH(fn, grid_for(n_episodes, ctx->threads, ctx->grid_evaluate[MAPF_POLICY_GROUPS]), ctx->threads, ctx->smem_base,
           stream, args);
    return MAPF_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// RTDP: value table, its Bellman update and its policy
// ---------------------------------------------------------------------------------------------------------------
static_assert(MAPF_VTABLE_EMPTY == VT_EMPTY && MAPF_VTABLE_REFUSED == VT_REFUSED, "value-table constants");

// The checks every value-table call makes: a one-word context and a well-formed table.
static int vtable_view(const mapf_ctx *ctx, const char *who, const mapf_vtable *t, VTableView *vt) {
    if (!ctx || !t || !t->keys || !t->values || !t->actions || !t->count)
        return fail(MAPF_ERR_INVALID, "%s: bad argument", who);
    if (t->capacity < 64 || (t->capacity & (t->capacity - 1)) != 0)
        return fail(MAPF_ERR_INVALID, "%s: capacity = %lld, must be a power of two >= 64", who, (long long)t->capacity);
    if (ctx->sp.words != 1)
        return fail(MAPF_ERR_UNSUPPORTED, "%s: the value table is keyed by one-word states; L**n = %d**%d needs two", who,
                    ctx->sp.L, ctx->sp.n);
    vt->keys = (const u64 *)t->keys;
    vt->values = t->values;
    vt->actions = t->actions;
    vt->mask = (u64)t->capacity - 1;
    return MAPF_OK;
}

static inline bool bad_states(int64_t B, const void *states) {
    return B < 0 || (B > 0 && (!states || ((uintptr_t)states & 7u) != 0));
}

extern "C" int mapf_rtdp_backup(const mapf_ctx *ctx, const void *states, int64_t B, const int32_t *group_of,
                                const double *hvalues, int64_t hvalues_len, const mapf_vtable *table, double gamma,
                                double *v_out, int32_t *a_out, void *stream) {
    VTableView vt = {};
    int rc = vtable_view(ctx, "mapf_rtdp_backup", table, &vt);
    if (rc) return rc;
    if (bad_states(B, states) || !group_of || !hvalues || (B > 0 && (!v_out || !a_out)))
        return fail(MAPF_ERR_INVALID, "mapf_rtdp_backup: bad argument");
    GroupLayout gl;
    u32 heads;
    rc = group_layout(ctx, "mapf_rtdp_backup", group_of, hvalues_len, &gl, &heads);
    if (rc) return rc;
    if (B == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    DevSpec sp = ctx->sp;
    // a warp takes G = max(1, 32 / nA) states per pass
    u32 G = ctx->sp.nA >= 32 ? 1u : (u32)(32 / ctx->sp.nA), rcp_nA = G > 1 ? (u32)(0xffffffffu / ctx->sp.nA + 1) : 0u;
    void *args[] = {&sp, &states, &B, &gl, &hvalues, &heads, &vt, &gamma, &G, &rcp_nA, &v_out, &a_out};
    const int64_t lanes = (B + G - 1) / G * 32;
    LAUNCH(ctx->ks.rtdp_backup, grid_for(lanes, ctx->threads, ctx->grid_rtdp), ctx->threads, ctx->smem_backup, stream,
           args);
    return MAPF_OK;
}

extern "C" int mapf_vtable_store(const mapf_ctx *ctx, const void *states, int64_t B, const double *v, const int32_t *a,
                                 const mapf_vtable *table, void *stream) {
    VTableView vt = {};
    int rc = vtable_view(ctx, "mapf_vtable_store", table, &vt);
    if (rc) return rc;
    if (bad_states(B, states) || (B > 0 && (!v || !a))) return fail(MAPF_ERR_INVALID, "mapf_vtable_store: bad argument");
    if (B == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    k_vtable_store<<<grid_for(B, 256, ctx->grid_plain), 256, 0, (cudaStream_t)stream>>>(
        (const u64 *)states, B, v, a, (u64 *)table->keys, table->values, table->actions, vt.mask, (u64 *)table->count);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

extern "C" int mapf_vtable_lookup(const mapf_ctx *ctx, const void *states, int64_t B, const int32_t *group_of,
                                  const double *hvalues, int64_t hvalues_len, const mapf_vtable *table, double *v_out,
                                  int32_t *a_out, void *stream) {
    VTableView vt = {};
    int rc = vtable_view(ctx, "mapf_vtable_lookup", table, &vt);
    if (rc) return rc;
    if (bad_states(B, states) || !group_of || !hvalues || (B > 0 && (!v_out || !a_out)))
        return fail(MAPF_ERR_INVALID, "mapf_vtable_lookup: bad argument");
    GroupLayout gl;
    u32 heads;
    rc = group_layout(ctx, "mapf_vtable_lookup", group_of, hvalues_len, &gl, &heads);
    if (rc) return rc;
    if (B == 0) return MAPF_OK;
    DeviceGuard g(ctx->device);
    DevSpec sp = ctx->sp;
    void *args[] = {&sp, &states, &B, &gl, &hvalues, &heads, &vt, &v_out, &a_out};
    LAUNCH(ctx->ks.vtable_lookup, grid_for(B, 256, ctx->grid_plain), 256, 0, stream, args);
    return MAPF_OK;
}

extern "C" int mapf_evaluate_table(const mapf_ctx *ctx, const mapf_vtable *table, const int32_t *group_of,
                                   const int32_t *tables, int64_t tables_len, int64_t n_episodes, int64_t max_steps,
                                   double gamma, uint64_t seed, uint64_t step_index0, int64_t episode_offset,
                                   void *scratch, double *ret, int32_t *length, uint8_t *outcome, uint8_t *conflict,
                                   void *stream) {
    VTableView vt = {};
    int rc = vtable_view(ctx, "mapf_evaluate_table", table, &vt);
    if (rc) return rc;
    if (!group_of || !tables || n_episodes < 0 || (n_episodes > 0 && (!scratch || !ret || !length || !outcome)))
        return fail(MAPF_ERR_INVALID, "mapf_evaluate_table: bad argument");
    if (max_steps < 1 || max_steps >= (1ll << 31))
        return fail(MAPF_ERR_INVALID, "mapf_evaluate_table: max_steps = %lld, must be in [1, 2**31)", (long long)max_steps);
    if (n_episodes > MAPF_LAUNCH_MAX_ENVS)
        return fail(MAPF_ERR_INVALID, "mapf_evaluate_table: at most 2**30 episodes per call");
    GroupLayout gl;
    u32 heads;
    rc = group_layout(ctx, "mapf_evaluate_table", group_of, tables_len, &gl, &heads);
    if (rc) return rc;
    if (!ctx->philox_ok)
        return fail(MAPF_ERR_UNSUPPORTED, "device-side sampling needs slip probabilities that add up to 1");
    if (n_episodes == 0) return MAPF_OK;
    DeviceGuard dg(ctx->device);
    CUDA_TRY(cudaMemsetAsync(scratch, 0, sizeof(u32), (cudaStream_t)stream));
    DevSpec sp = ctx->sp;
    PhiloxKeys keys = make_keys(seed);
    u32 E = (u32)n_episodes, T = (u32)max_steps;
    u64 st = step_index0, e0 = (u64)episode_offset;
    void *args[] = {&sp, &keys, &tables, &gl, &vt, &E, &T, &gamma, &st, &e0, &scratch, &ret, &length, &outcome, &conflict};
    LAUNCH(ctx->ks.evaluate_table, grid_for(n_episodes, ctx->threads, ctx->grid_evaluate_table), ctx->threads,
           ctx->smem_base, stream, args);
    return MAPF_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// host-buffer step: H2D, step, D2H in two pipelined halves on the context's own streams
// ---------------------------------------------------------------------------------------------------------------
// `keep` != NULL (mapf_step_host_resident): the envs' states live in DEVICE memory at `keep`; they are read from there
// instead of from the host pointer `states` (ignored) and overwritten in place with the next states by the KEEP kernels.
static int step_host_impl(mapf_ctx *ctx, const void *states, void *keep, const int32_t *actions, int64_t B,
                          const double *uniforms, uint64_t seed, uint64_t step_index, int64_t env_offset,
                          uint32_t options, void *next_states, double *reward, double *prob, uint8_t *done,
                          uint8_t *collision) {
    if (!ctx || B < 0 || (B > 0 && ((!states && !keep) || !actions || !next_states || !reward || !prob || !done ||
                                     (!collision && !(options & MAPF_OPT_COMPACT)))))
        return fail(MAPF_ERR_INVALID, "%s: bad argument", keep ? "mapf_step_host_resident" : "mapf_step_host");
    if (keep && B > 0) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, keep) != cudaSuccess || at.type != cudaMemoryTypeDevice || at.device != ctx->device) {
            cudaGetLastError();
            return fail(MAPF_ERR_INVALID, "mapf_step_host_resident: states_dev must be device memory of the context's GPU");
        }
    }
    const bool compact = (options & MAPF_OPT_COMPACT) != 0;
    const size_t rw = compact ? 1 : 8;  // bytes of a reward / reward code
    if (B == 0) return MAPF_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    DeviceGuard g(ctx->device);
    const int n = ctx->sp.n;
    const size_t sw = (size_t)ctx->sp.words * 8;
    for (int i = 0; i < MAPF_HOST_STREAMS; ++i)
        if (!ctx->hs[i]) CUDA_TRY(cudaStreamCreateWithFlags(&ctx->hs[i], cudaStreamNonBlocking));
    // Small batches (the scalar MapfEnv.step is B = 1): the fixed cost of eight staged copies dwarfs the work.  Pack
    // the inputs into the context's page-locked scratch, run the kernel directly on its device mapping (zero copy),
    // unpack: one launch and one synchronisation.
    if (B <= MAPF_SMALL_HOST_BATCH) {
        const size_t cap = MAPF_SMALL_HOST_BATCH;
        const size_t o_s = 0, o_a = o_s + 16 * cap, o_u = o_a + 4 * cap, o_ns = o_u + 8 * MAPF_MAXN * cap,
                     o_r = o_ns + 16 * cap, o_p = o_r + 8 * cap, o_d = o_p + 8 * cap, o_c = o_d + cap, total = o_c + cap;
        if (!ctx->h_small) {
            CUDA_TRY(cudaHostAlloc((void **)&ctx->h_small, total, cudaHostAllocMapped));
            CUDA_TRY(cudaHostGetDevicePointer((void **)&ctx->h_small_dev, ctx->h_small, 0));
        }
        unsigned char *h = ctx->h_small, *d = ctx->h_small_dev;
        if (!keep) memcpy(h + o_s, states, sw * B);
        memcpy(h + o_a, actions, 4 * (size_t)B);
        if (uniforms) memcpy(h + o_u, uniforms, (size_t)n * 8 * B);
        int rc = launch_step(ctx, keep ? keep : d + o_s, (const int32_t *)(d + o_a), B,
                             uniforms ? (const double *)(d + o_u) : nullptr, seed, step_index, env_offset, options, d + o_ns,
                             (double *)(d + o_r), (double *)(d + o_p), d + o_d, d + o_c, ctx->hs[0], 0, keep);
        if (rc) return rc;
        CUDA_TRY(cudaStreamSynchronize(ctx->hs[0]));
        memcpy(next_states, h + o_ns, sw * B);
        memcpy(reward, h + o_r, rw * (size_t)B);
        memcpy(prob, h + o_p, 8 * (size_t)B);
        memcpy(done, h + o_d, (size_t)B);
        if (!compact) memcpy(collision, h + o_c, (size_t)B);
        return MAPF_OK;
    }
    // Zero-copy path: when every buffer is page-locked host memory that the device can address (cudaHostAlloc /
    // cudaHostRegister, e.g. torch's pin_memory()), ONE launch of the step kernel reads the inputs and writes the
    // results straight over PCIe -- both directions stream concurrently, with no staging copies and no per-copy
    // driver calls.  Otherwise fall back to staged copies below.
    {
        const void *host_in[3] = {states, actions, uniforms};
        void *host_out[5] = {next_states, reward, prob, done, collision};
        void *dev_in[3] = {nullptr, nullptr, nullptr}, *dev_out[5];
        // (Chunked cudaMemcpyAsync pipelines were measured against this zero-copy launch on 2**20 envs and lost: 8 chunks
        // over 4 streams 1.29e9 env-steps/s, two halves 1.48e9, zero copy 1.70e9 -- the 7 driver calls per chunk cost
        // more than the copy engines gain.)
        bool mapped = true;
#ifdef MAPF_TUNING
        if (const char *e = getenv("MAPF_HOST_MODE")) mapped = atoi(e) == 0;  // 0 zero-copy, 1 staged copies
#endif
        for (int i = keep ? 1 : 0; i < 3 && mapped; ++i) {
            if (!host_in[i]) continue;
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, host_in[i]) != cudaSuccess || at.type != cudaMemoryTypeHost ||
                !at.devicePointer) { cudaGetLastError(); mapped = false; break; }
            dev_in[i] = at.devicePointer;
        }
        for (int i = 0; i < 5 && mapped; ++i) {
            dev_out[i] = nullptr;
            if (!host_out[i]) continue;  // collision in compact mode
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, host_out[i]) != cudaSuccess || at.type != cudaMemoryTypeHost ||
                !at.devicePointer) { cudaGetLastError(); mapped = false; break; }
            dev_out[i] = at.devicePointer;
        }
        if (mapped) {
            // over PCIe fewer, longer sequential streams move more bytes: 2**20 envs with 296 / 148 / 74 / 37 CTAs reach
            // 1.61 / 1.70 / 1.74 / 1.75e9 env-steps/s (profiles/r02_ablations.txt)
            int host_grid = B >= (1 << 18) ? (ctx->info.sm_count + 3) / 4 : ctx->info.sm_count;
#ifdef MAPF_TUNING
            if (const char *e = getenv("MAPF_HOST_GRID")) host_grid = atoi(e);
#endif
            int rc = launch_step(ctx, keep ? keep : dev_in[0], (const int32_t *)dev_in[1], B, (const double *)dev_in[2], seed,
                                 step_index, env_offset, options, dev_out[0], (double *)dev_out[1], (double *)dev_out[2],
                                 (uint8_t *)dev_out[3], (uint8_t *)dev_out[4], ctx->hs[0], host_grid, keep);
            if (rc) return rc;
            CUDA_TRY(cudaStreamSynchronize(ctx->hs[0]));
            return MAPF_OK;
        }
    }
    // per-env device bytes: state in, action, uniforms, state out, reward, prob, done, collision
    // (resident states: the kernels of the two halves work on disjoint env ranges of `keep`, in place)
    const size_t per_env = sw + 4 + (uniforms ? (size_t)n * 8 : 0) + sw + 8 + 8 + 1 + 1;
    const size_t need = per_env * (size_t)B + 8 * 256;
    if (need > ctx->d_stage_bytes) {
        if (ctx->d_stage) cudaFree(ctx->d_stage);
        ctx->d_stage = nullptr;
        ctx->d_stage_bytes = 0;
        CUDA_TRY(cudaMalloc(&ctx->d_stage, need));
        ctx->d_stage_bytes = need;
    }
    auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
    unsigned char *p = ctx->d_stage;
    unsigned char *d_s = p; p += align(sw * B);
    unsigned char *d_a = p; p += align(4 * (size_t)B);
    unsigned char *d_u = p; p += uniforms ? align((size_t)n * 8 * B) : 0;
    unsigned char *d_ns = p; p += align(sw * B);
    unsigned char *d_r = p; p += align(8 * (size_t)B);
    unsigned char *d_p = p; p += align(8 * (size_t)B);
    unsigned char *d_d = p; p += align((size_t)B);
    unsigned char *d_c = p;
    // chunk boundaries are even (128-bit I/O)
    const int parts = B >= (1 << 16) ? 2 : 1;  // pageable buffers: two pipelined halves
    for (int h = 0; h < parts; ++h) {
        const int64_t b0 = (B * h / parts) & ~(int64_t)1, b1 = h + 1 == parts ? B : ((B * (h + 1) / parts) & ~(int64_t)1),
                      nb = b1 - b0;
        if (nb <= 0) continue;
        cudaStream_t st = ctx->hs[h % MAPF_HOST_STREAMS];
        if (!keep)
            CUDA_TRY(cudaMemcpyAsync(d_s + sw * b0, (const unsigned char *)states + sw * b0, sw * nb, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(d_a + 4 * b0, (const unsigned char *)actions + 4 * b0, 4 * nb, cudaMemcpyHostToDevice, st));
        if (uniforms)
            CUDA_TRY(cudaMemcpyAsync(d_u + (size_t)n * 8 * b0, (const unsigned char *)uniforms + (size_t)n * 8 * b0,
                                     (size_t)n * 8 * nb, cudaMemcpyHostToDevice, st));
        unsigned char *k0 = keep ? (unsigned char *)keep + sw * b0 : nullptr;
        int rc = launch_step(ctx, keep ? k0 : d_s + sw * b0, (const int32_t *)(d_a + 4 * b0), nb,
                             uniforms ? (const double *)(d_u + (size_t)n * 8 * b0) : nullptr, seed, step_index,
                             env_offset + b0, options, d_ns + sw * b0, (double *)(d_r + rw * b0), (double *)(d_p + 8 * b0),
                             d_d + b0, d_c + b0, st, 0, k0);
        if (rc) return rc;
        CUDA_TRY(cudaMemcpyAsync((unsigned char *)next_states + sw * b0, d_ns + sw * b0, sw * nb, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync((unsigned char *)reward + rw * b0, d_r + rw * b0, rw * nb, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync((unsigned char *)prob + 8 * b0, d_p + 8 * b0, 8 * nb, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(done + b0, d_d + b0, nb, cudaMemcpyDeviceToHost, st));
        if (!compact) CUDA_TRY(cudaMemcpyAsync(collision + b0, d_c + b0, nb, cudaMemcpyDeviceToHost, st));
    }
    for (int h = 0; h < MAPF_HOST_STREAMS; ++h) CUDA_TRY(cudaStreamSynchronize(ctx->hs[h]));
    return MAPF_OK;
}

extern "C" int mapf_step_host(mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B,
                              const double *uniforms, uint64_t seed, uint64_t step_index, int64_t env_offset,
                              uint32_t options, void *next_states, double *reward, double *prob, uint8_t *done,
                              uint8_t *collision) {
    if (B > 0 && !states) return fail(MAPF_ERR_INVALID, "mapf_step_host: bad argument");
    return step_host_impl(ctx, states, nullptr, actions, B, uniforms, seed, step_index, env_offset, options, next_states,
                          reward, prob, done, collision);
}

extern "C" int mapf_step_host_resident(mapf_ctx *ctx, void *states_dev, const int32_t *actions, int64_t B,
                                       const double *uniforms, uint64_t seed, uint64_t step_index, int64_t env_offset,
                                       uint32_t options, void *next_states, double *reward, double *prob, uint8_t *done,
                                       uint8_t *collision) {
    if (B > 0 && (!states_dev || (ctx && states_misaligned(ctx->sp.words, states_dev))))
        return fail(MAPF_ERR_INVALID, "mapf_step_host_resident: bad argument");
    return step_host_impl(ctx, nullptr, states_dev, actions, B, uniforms, seed, step_index, env_offset, options, next_states,
                          reward, prob, done, collision);
}

// ---------------------------------------------------------------------------------------------------------------
// on-disk formats (SURVEY.md 8f row 4): MovingAI .map text parsed on the device, .scen text on the host
// ---------------------------------------------------------------------------------------------------------------
#include "mapf_parse.cuh"

// int() of one tab-separated scenario field: optional surrounding whitespace, optional sign, decimal digits
static bool parse_int_field(const char *b, const char *e, long long *out) {
    while (b < e && ((unsigned char)*b <= 32)) ++b;
    while (e > b && ((unsigned char)e[-1] <= 32)) --e;
    if (b >= e) return false;
    bool neg = false;
    if (*b == '+' || *b == '-') { neg = *b == '-'; ++b; }
    if (b >= e) return false;
    long long v = 0;
    for (; b < e; ++b) {
        if (*b == '_' && b + 1 < e) continue;  // Python accepts 1_000
        if (*b < '0' || *b > '9') return false;
        v = v * 10 + (*b - '0');
        if (v > (1ll << 40)) return false;
    }
    *out = neg ? -v : v;
    return true;
}

// parse_scen_file (utils.py:8-30): skip the "version" line; every further line must have exactly nine tab-separated
// fields (the reference's tuple unpacking raises ValueError otherwise); fields 4..7 are used AS (row, col) pairs in
// file order; stops after n_agents lines or at the end of the file (`n_agents` is truncated, utils.py:123).
static int parse_scen_text(const char *text, int64_t len, int n_agents, int32_t *start_rc, int32_t *goal_rc, int *n_found) {
    int64_t p = 0;
    auto next_line = [&](int64_t &b, int64_t &e) -> bool {  // [b, e) without the terminator; universal newlines
        if (p >= len) return false;
        b = p;
        while (p < len && text[p] != '\n' && text[p] != '\r') ++p;
        e = p;
        if (p < len) { if (text[p] == '\r' && p + 1 < len && text[p + 1] == '\n') p += 2; else p += 1; }
        return true;
    };
    int64_t b, e;
    if (!next_line(b, e)) return fail(MAPF_ERR_INVALID, "scenario text is empty (StopIteration in the reference)");
    int got = 0;
    while (got < n_agents && next_line(b, e)) {
        int64_t fb[10];
        int nf = 0;
        fb[0] = b;
        for (int64_t q = b; q < e; ++q)
            if (text[q] == '\t') { if (nf < 9) fb[++nf] = q + 1; else ++nf; }
        const int fields = nf + 1;
        if (fields != 9)
            return fail(MAPF_ERR_INVALID, "scenario line %d has %d tab-separated fields, expected 9", got + 2, fields);
        fb[9] = e + 1;
        long long v[4];
        for (int k = 0; k < 4; ++k)
            if (!parse_int_field(text + fb[4 + k], text + fb[5 + k] - 1, &v[k]))
                return fail(MAPF_ERR_INVALID, "scenario line %d: field %d is not an integer", got + 2, 4 + k);
        start_rc[2 * got] = (int32_t)v[0]; start_rc[2 * got + 1] = (int32_t)v[1];
        goal_rc[2 * got] = (int32_t)v[2]; goal_rc[2 * got + 1] = (int32_t)v[3];
        ++got;
    }
    *n_found = got;
    return MAPF_OK;
}

extern "C" int mapf_parse_scen_text(const char *scen_text, int64_t scen_len, int32_t n_agents, int32_t *start_rc,
                                    int32_t *goal_rc, int32_t *n_found) {
    if (!scen_text || scen_len < 0 || n_agents < 1 || !start_rc || !goal_rc || !n_found)
        return fail(MAPF_ERR_INVALID, "mapf_parse_scen_text: bad argument");
    int found = 0;
    const int rc = parse_scen_text(scen_text, scen_len, n_agents, start_rc, goal_rc, &found);
    *n_found = found;
    return rc;
}

extern "C" int mapf_parse_map_text(const char *map_text, int64_t map_len, int device, int32_t *height, int32_t *width,
                                   uint8_t *obstacles, int64_t obstacles_cap) {
    if (!map_text || map_len < 0 || !height || !width) return fail(MAPF_ERR_INVALID, "mapf_parse_map_text: bad argument");
    if (map_len > (64ll << 20)) return fail(MAPF_ERR_UNSUPPORTED, "map text of %lld bytes: at most 64 MiB", (long long)map_len);
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev < 1 || device < 0 || device >= n_dev)
        return fail(MAPF_ERR_NO_DEVICE, "CUDA device %d is not available (%d devices): there is no CPU fallback", device, n_dev);
    DeviceGuard guard(device);
    if (!guard.ok) return fail(MAPF_ERR_CUDA, "cannot select device %d", device);
    const u32 len = (u32)map_len;
    // one allocation: text | line_start[len + 2] | row_begin[len + 1] | row_len[len + 1] | obstacles[len] | header
    const size_t o_text = 0, o_ls = (o_text + len + 15) & ~(size_t)15, o_rb = o_ls + 4 * ((size_t)len + 2),
                 o_rl = o_rb + 4 * ((size_t)len + 1), o_ob = o_rl + 4 * ((size_t)len + 1),
                 o_hdr = (o_ob + len + 15) & ~(size_t)15, total = o_hdr + sizeof(ParsedMapHeader);
    unsigned char *d = nullptr;
    CUDA_TRY(cudaMalloc(&d, total));
    struct Free { unsigned char *p; ~Free() { cudaFree(p); } } guard_free{d};
    if (len) CUDA_TRY(cudaMemcpy(d + o_text, map_text, len, cudaMemcpyHostToDevice));
    k_parse_map<<<1, PARSE_THREADS>>>(d + o_text, len, (u32 *)(d + o_ls), (u32 *)(d + o_rb), (u32 *)(d + o_rl), d + o_ob,
                                      (ParsedMapHeader *)(d + o_hdr));
    CUDA_TRY(cudaGetLastError());
    ParsedMapHeader hdr;
    CUDA_TRY(cudaMemcpy(&hdr, d + o_hdr, sizeof(hdr), cudaMemcpyDeviceToHost));
    if (hdr.H < 1 || hdr.W < 1)
        return fail(MAPF_ERR_INVALID, "map text has %d lines: no grid rows behind the 4 header lines", hdr.n_lines);
    if (hdr.bad_pos != 0xffffffffu) {  // CHAR_TO_CELL[char] raises KeyError (grid.py:21)
        if (hdr.bad_char >= 32 && hdr.bad_char < 127) return fail(MAPF_ERR_KEY, "'%c'", (int)hdr.bad_char);
        return fail(MAPF_ERR_KEY, "'\\x%02x'", hdr.bad_char);
    }
    if (hdr.ragged)
        return fail(MAPF_ERR_INVALID, "grid row %d is not %d cells wide like row 0", hdr.ragged - 1, hdr.W);
    *height = hdr.H;
    *width = hdr.W;
    if (obstacles) {
        if (obstacles_cap < (int64_t)hdr.H * hdr.W)
            return fail(MAPF_ERR_INVALID, "obstacle buffer of %lld bytes for a %dx%d grid", (long long)obstacles_cap, hdr.H, hdr.W);
        CUDA_TRY(cudaMemcpy(obstacles, d + o_ob, (size_t)hdr.H * hdr.W, cudaMemcpyDeviceToHost));
    }
    return MAPF_OK;
}

extern "C" int mapf_ctx_create_from_text(const char *map_text, int64_t map_len, const char *scen_text, int64_t scen_len,
                                         int32_t n_agents, double fail_prob, double reward_of_clash, double reward_of_goal,
                                         double reward_of_living, int32_t criterion, int device, mapf_ctx **out) {
    if (!map_text || !scen_text || map_len < 0 || scen_len < 0 || !out)
        return fail(MAPF_ERR_INVALID, "mapf_ctx_create_from_text: bad argument");
    *out = nullptr;
    if (n_agents < 1) return fail(MAPF_ERR_INVALID, "n_agents = %d", n_agents);
    int32_t H = 0, W = 0;
    std::vector<uint8_t> obstacles((size_t)map_len + 1);
    int rc = mapf_parse_map_text(map_text, map_len, device, &H, &W, obstacles.data(), (int64_t)obstacles.size());
    if (rc) return rc;
    const int want = n_agents < 4096 ? n_agents : 4096;
    std::vector<int32_t> start_rc(2 * (size_t)want), goal_rc(2 * (size_t)want);
    int found = 0;
    rc = parse_scen_text(scen_text, scen_len, want, start_rc.data(), goal_rc.data(), &found);
    if (rc) return rc;
    if (found < 1) return fail(MAPF_ERR_INVALID, "the scenario holds no agent");
    mapf_spec spec;
    memset(&spec, 0, sizeof(spec));
    spec.height = H; spec.width = W;
    spec.obstacles = obstacles.data();
    spec.n_agents = found;  // n_agents = len(agents_goals) (utils.py:123)
    spec.start_rc = start_rc.data();
    spec.goal_rc = goal_rc.data();
    spec.fail_prob = fail_prob;
    spec.reward_of_clash = reward_of_clash; spec.reward_of_goal = reward_of_goal; spec.reward_of_living = reward_of_living;
    spec.criterion = criterion;
    return mapf_ctx_create(&spec, device, out);
}

extern "C" int mapf_ctx_grid(const mapf_ctx *ctx, int32_t *height, int32_t *width, uint8_t *obstacles, int32_t *start_rc,
                             int32_t *goal_rc) {
    if (!ctx) return fail(MAPF_ERR_INVALID, "mapf_ctx_grid: NULL context");
    const int H = ctx->sp.H, W = ctx->sp.Wd;
    if (height) *height = H;
    if (width) *width = W;
    if (obstacles) {
        memset(obstacles, 1, (size_t)H * W);
        for (int i = 0; i < ctx->sp.L; ++i)
            obstacles[(size_t)(ctx->h_cell_rc[i] >> 16) * W + (ctx->h_cell_rc[i] & 0xffffu)] = 0;
    }
    for (int i = 0; i < ctx->sp.n; ++i) {
        const u32 s = ctx->h_cell_rc[ctx->sp.start[i]], g = ctx->h_cell_rc[ctx->sp.goal[i]];
        if (start_rc) { start_rc[2 * i] = (int32_t)(s >> 16); start_rc[2 * i + 1] = (int32_t)(s & 0xffffu); }
        if (goal_rc) { goal_rc[2 * i] = (int32_t)(g >> 16); goal_rc[2 * i + 1] = (int32_t)(g & 0xffffu); }
    }
    return MAPF_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// heterogeneous batches (SURVEY.md 8f row 4): one launch steps envs of several specs
// ---------------------------------------------------------------------------------------------------------------
struct mapf_group {
    int device = 0;
    int n = 0, words = 0, n_specs = 0;
    int threads = 512, grid = 0;
    int64_t B = 0;
    u32 spec_off = 0;
    size_t smem = 0;
    bool philox_ok = true;
    const void *fn_philox = nullptr, *fn_tape = nullptr;
    DevSpec *d_specs = nullptr;
    u32 *d_seg = nullptr;               // seg_begin[n_specs + 1]
    std::vector<int64_t> seg_begin;
};

extern "C" void mapf_group_destroy(mapf_group *g) {
    if (!g) return;
    {
        DeviceGuard guard(g->device);
        cudaFree(g->d_specs);
        cudaFree(g->d_seg);
    }
    delete g;
}

extern "C" int mapf_group_create(mapf_ctx *const *ctxs, const int64_t *env_counts, int32_t n_specs, mapf_group **out) {
    if (!ctxs || !env_counts || n_specs < 1 || !out) return fail(MAPF_ERR_INVALID, "mapf_group_create: bad argument");
    *out = nullptr;
    for (int i = 0; i < n_specs; ++i)
        if (!ctxs[i] || env_counts[i] < 0) return fail(MAPF_ERR_INVALID, "mapf_group_create: bad spec %d", i);
    const mapf_ctx *c0 = ctxs[0];
    size_t smem_max = 0;
    int64_t B = 0;
    bool philox_ok = true;
    for (int i = 0; i < n_specs; ++i) {
        const mapf_ctx *c = ctxs[i];
        if (c->device != c0->device) return fail(MAPF_ERR_INVALID, "spec %d lives on device %d, spec 0 on %d", i, c->device, c0->device);
        if (c->sp.n != c0->sp.n || c->sp.words != c0->sp.words)
            return fail(MAPF_ERR_UNSUPPORTED,
                        "spec %d has %d agents and %d-word states, spec 0 has %d and %d: one group = one agent count and "
                        "state width (step other specs with their own mapf_step)",
                        i, c->sp.n, c->sp.words, c0->sp.n, c0->sp.words);
        if (!c->sp.lut_smem)
            return fail(MAPF_ERR_UNSUPPORTED, "spec %d: its move table is not staged in shared memory (too many cells); step it "
                                              "with its own mapf_step", i);
        if (c->sp.smem_window != c0->sp.smem_window) return fail(MAPF_ERR_INVALID, "specs were built for different shared-memory windows");
        if (c->smem_base > smem_max) smem_max = c->smem_base;
        philox_ok = philox_ok && c->philox_ok;
        B += env_counts[i];
    }
    if (B >= (1ll << 31)) return fail(MAPF_ERR_UNSUPPORTED, "%lld envs: a group holds fewer than 2**31", (long long)B);
    mapf_group *g = new (std::nothrow) mapf_group();
    if (!g) return fail(MAPF_ERR_INVALID, "out of host memory");
    g->device = c0->device; g->n = c0->sp.n; g->words = c0->sp.words; g->n_specs = n_specs; g->B = B;
    g->philox_ok = philox_ok;
    g->fn_philox = c0->ks.step_group_philox;
    g->fn_tape = c0->ks.step_group_tape;
    g->spec_off = (u32)((smem_max + 15) & ~(size_t)15);
    g->smem = g->spec_off + ((sizeof(DevSpec) + 15) & ~(size_t)15);
    std::vector<DevSpec> specs(n_specs);
    std::vector<u32> seg((size_t)n_specs + 1);
    g->seg_begin.resize((size_t)n_specs + 1);
    int64_t at = 0;
    for (int i = 0; i < n_specs; ++i) {
        specs[i] = ctxs[i]->sp;
        g->seg_begin[i] = at;
        seg[i] = (u32)at;
        at += env_counts[i];
    }
    g->seg_begin[n_specs] = at;
    seg[n_specs] = (u32)at;
    DeviceGuard guard(g->device);
#define GRP_TRY(expr)                                                                                  \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess) {                                                                       \
            int _rc = fail(MAPF_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            mapf_group_destroy(g);                                                                     \
            return _rc;                                                                                \
        }                                                                                              \
    } while (0)
    if (!g->fn_philox || !g->fn_tape) { mapf_group_destroy(g); return fail(MAPF_ERR_UNSUPPORTED, "no grouped step kernel for this spec"); }
    GRP_TRY(cudaMalloc(&g->d_specs, sizeof(DevSpec) * (size_t)n_specs));
    GRP_TRY(cudaMemcpy(g->d_specs, specs.data(), sizeof(DevSpec) * (size_t)n_specs, cudaMemcpyHostToDevice));
    GRP_TRY(cudaMalloc(&g->d_seg, sizeof(u32) * seg.size()));
    GRP_TRY(cudaMemcpy(g->d_seg, seg.data(), sizeof(u32) * seg.size(), cudaMemcpyHostToDevice));
    int grid_p = 0, grid_t = 0;
    cudaDeviceProp prop;
    GRP_TRY(cudaGetDeviceProperties(&prop, g->device));
    if (g->smem > (size_t)prop.sharedMemPerBlockOptin) {
        mapf_group_destroy(g);
        return fail(MAPF_ERR_UNSUPPORTED, "the group's largest image needs %zu B of shared memory", g->smem);
    }
    for (const void *fn : {g->fn_philox, g->fn_tape})
        if (int rc = raise_smem_cap(g->device, fn, g->smem)) { mapf_group_destroy(g); return rc; }
    int rc = occupancy_grid(g->fn_philox, g->threads, g->smem, c0->info.sm_count, &grid_p);
    if (!rc) rc = occupancy_grid(g->fn_tape, g->threads, g->smem, c0->info.sm_count, &grid_t);
    if (rc) { mapf_group_destroy(g); return rc; }
    g->grid = grid_p < grid_t ? grid_p : grid_t;
    *out = g;
    return MAPF_OK;
}

extern "C" int mapf_group_step(const mapf_group *g, const void *states, const int32_t *actions, const double *uniforms,
                               uint64_t seed, uint64_t step_index, int64_t env_offset, uint32_t options, void *next_states,
                               double *reward, double *prob, uint8_t *done, uint8_t *collision, void *stream) {
    if (!g) return fail(MAPF_ERR_INVALID, "mapf_group_step: NULL group");
    // k_step_group writes the default result layout and takes no launch-shape option: a compact-sized reward buffer
    // would be overrun by its 8-byte stores
    if (options & ~(uint32_t)MAPF_OPT_AUTO_RESET)
        return fail(MAPF_ERR_UNSUPPORTED, "mapf_group_step: options = %u, only MAPF_OPT_AUTO_RESET is supported (step "
                                          "with mapf_step for the compact layout)", options);
    if (g->B == 0) return MAPF_OK;
    if (!states || !actions || !next_states || !reward || !prob || !done || !collision ||
        states_misaligned(g->words, states) || states_misaligned(g->words, next_states))
        return fail(MAPF_ERR_INVALID, "mapf_group_step: NULL buffer");
    if (!uniforms && !g->philox_ok)
        return fail(MAPF_ERR_UNSUPPORTED, "device-side sampling needs slip probabilities that add up to 1; pass uniforms");
    DeviceGuard guard(g->device);
    PhiloxKeys keys = make_keys(seed);
    const DevSpec *specs = g->d_specs;
    const u32 *seg = g->d_seg;
    u32 n_specs = (u32)g->n_specs, nb = (u32)g->B, spec_off = g->spec_off, op = options;
    u64 st = step_index, e0 = (u64)env_offset;
    void *args[] = {&specs, &seg, &n_specs, &nb, &spec_off, &keys, &states, &actions, &uniforms, &st, &e0, &op, &next_states,
                    &reward, &prob, &done, &collision};
    // every CTA owns a contiguous range of envs; small batches get one CTA per 2 * threads envs
    const int64_t want = (g->B + 2 * g->threads - 1) / (2 * g->threads);
    const int grid = (int)(want < g->grid ? want : g->grid);
    // programmatic stream serialization (see launch_step): this launch may begin, up to its griddepcontrol.wait, while
    // the previous kernel of the stream is still draining
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(g->threads);
    cfg.dynamicSmemBytes = g->smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelExC(&cfg, uniforms ? g->fn_tape : g->fn_philox, args);
    if (e != cudaSuccess) return fail(MAPF_ERR_CUDA, "launch k_step_group: %s", cudaGetErrorString(e));
    return MAPF_OK;
}

extern "C" int64_t mapf_group_size(const mapf_group *g) { return g ? g->B : -1; }
