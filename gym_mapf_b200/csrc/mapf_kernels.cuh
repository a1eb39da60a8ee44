// mapf_kernels.cuh -- the sm_100a kernels of the joint-transition engine.
//
// Mapping: one thread per emitted unit -- one env-step in step/rollout mode, one P[s][a] record in
// expand mode.  All per-agent loops are unrolled over the template parameter N, so an agent's cell, move-table
// entry and outcome digit live in registers.  The per-(cell, action) move table is staged in shared memory by one
// bulk asynchronous copy (TMA engine) per CTA.
//
// Reference citations are file:line relative to /root/reference/gym_mapf/envs/.
#pragma once
#include "mapf_device.cuh"

// Timeline builds only (-DMAPF_TRACE, tools/trace_step.py): thread 0 of every CTA of the Philox-mode k_step stamps
// %globaltimer at its phase boundaries into the buffer passed in place of the (unused) `uniforms` pointer:
// buf[0] = next free slot; slot = {tag << 48 | (step & 0xffff) << 32 | smid << 16 | blockIdx, nanoseconds}.
#ifdef MAPF_TRACE
__device__ __forceinline__ void trace_stamp(const double *buf, u64 step, u32 tag) {
    if (threadIdx.x != 0 || buf == nullptr) return;
    u64 *b = reinterpret_cast<u64 *>(const_cast<double *>(buf));
    u64 t;
    u32 smid;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    const u64 slot = atomicAdd(reinterpret_cast<unsigned long long *>(b), 1ull);
    if (slot < (1ull << 20)) {
        b[2 + 2 * slot] = ((u64)tag << 48) | ((step & 0xffffull) << 32) | ((u64)smid << 16) | (u64)blockIdx.x;
        b[3 + 2 * slot] = t;
    }
}
#define TRACE(tag) trace_stamp(uniforms, step, tag)
#else
#define TRACE(tag)
#endif
#ifndef MAPF_PREFETCH_ITEMS
#define MAPF_PREFETCH_ITEMS 1
#endif
#ifndef MAPF_MAX_THREADS
#define MAPF_MAX_THREADS 512  // largest CTA the hot kernels are launched with
#endif
// Register budget of the step kernel: up to 6 agents everything fits 64 registers (2 CTAs of 512 or 4 of 256
// threads per SM, measured best on the 4-agent workload); more agents get the full 128.
#ifndef MAPF_MIN_BLOCKS
#define MAPF_MIN_BLOCKS(N) ((N) <= 6 ? 2 : 1)
#endif

// =====================================================================================================
// Move-table construction from the obstacle bitmap (ctx creation; not a hot kernel)
// =====================================================================================================
// colbits: per column c, wpc 32-bit words; bit r of the column is 1 when cell (r, c) is FREE.
// colbase: number of free cells in columns < c, i.e. the id of the first free cell of column c
//          (column-major numbering: grid.py:37-40, mapf_env.py:142-143).
// The whole bitmap is staged in shared memory; one thread per grid position.
struct BitmapView {
    const u32 *bits;
    const u32 *base;
    int H, W, wpc;
};

__device__ __forceinline__ bool bm_free(const BitmapView &bm, int r, int c) {
    return (bm.bits[c * bm.wpc + (r >> 5)] >> (r & 31)) & 1u;
}

__device__ __forceinline__ int bm_rank(const BitmapView &bm, int r, int c) {
    int id = (int)bm.base[c];
    const u32 *col = bm.bits + c * bm.wpc;
    for (int w = 0; w < (r >> 5); ++w) id += __popc(col[w]);
    id += __popc(col[r >> 5] & ((1u << (r & 31)) - 1u));
    return id;
}

// execute_up/down/right/left/stay + stay_if_hit_obstacle (mapf_env.py:43-84): clamp to the grid, obstacle = stay
__device__ __forceinline__ void bm_move(const BitmapView &bm, int r, int c, int d, int &nr, int &nc) {
    int tr = r, tc = c;
    if (d == 1) tr = max(0, r - 1);
    else if (d == 3) tr = min(bm.H - 1, r + 1);
    else if (d == 2) tc = min(bm.W - 1, c + 1);
    else if (d == 4) tc = max(0, c - 1);
    bool ok = (d == 0) || bm_free(bm, tr, tc);
    nr = ok ? tr : r;
    nc = ok ? tc : c;
}

// The merge patterns that can occur, as 9-bit triples (mask of slot 0 | mask of slot 1 << 3 | mask of slot 2 << 6)
// of candidate bits {intended = 1, right = 2, left = 4}; the index of a triple is its pattern id.
struct PatternList {
    u32 triple[MAPF_MAX_PATTERNS];
    int count;
};

// single_agent_movements (mapf_env.py:163-184) for one (cell, action): candidates [intended, right, left],
// zero-probability candidates dropped (cand_mask), equal destinations merged into the first occurrence.
__device__ __forceinline__ u64 bm_entry(const BitmapView &bm, int r, int c, int a, int cand_mask,
                                        const PatternList &pats) {
    // POSSIBILITIES (__init__.py:19-25): right/left slip of STAY,UP,RIGHT,DOWN,LEFT
    const int slip_r[5] = {0, 2, 3, 4, 1};
    const int slip_l[5] = {0, 4, 1, 2, 3};
    int dir[3] = {a, slip_r[a], slip_l[a]};
    u32 dest[3] = {0, 0, 0}, mask[3] = {0, 0, 0};
    int k = 0;
    for (int j = 0; j < 3; ++j) {
        if (!((cand_mask >> j) & 1)) continue;
        int nr, nc;
        bm_move(bm, r, c, dir[j], nr, nc);
        u32 id = (u32)bm_rank(bm, nr, nc);
        int at = -1;
        for (int q = 0; q < k; ++q)
            if (dest[q] == id && at < 0) at = q;
        if (at >= 0) mask[at] |= 1u << j;
        else { dest[k] = id; mask[k] = 1u << j; ++k; }
    }
    for (int q = k; q < 3; ++q) dest[q] = dest[0];
    const u32 triple = mask[0] | (mask[1] << 3) | (mask[2] << 6);
    u32 pid = 0;
    for (int q = 0; q < pats.count; ++q)
        if (pats.triple[q] == triple) pid = (u32)q;
    return (u64)dest[0] | ((u64)dest[1] << 16) | ((u64)dest[2] << 32) | ((u64)(pid * MAPF_PAT_STRIDE) << 48) | ((u64)k << 56);
}

// shared-window address of a kernel's dynamic shared memory (context creation; see DevSpec::smem_window)
static __global__ void k_probe_smem(u32 *out) {
    extern __shared__ __align__(16) unsigned char probe_smem[];
    if (threadIdx.x == 0) *out = smem_u32(probe_smem);
}

struct GoalList {
    u16 cell[16];
    int n;
};

static __global__ void k_build_moves(const u32 *__restrict__ colbits, const u32 *__restrict__ colbase, int H, int W, int wpc,
                              int cand_mask, PatternList pats, GoalList goals, u64 *__restrict__ lut,
                              u32 *__restrict__ cell_rc) {
    extern __shared__ u32 bm_smem[];
    u32 *s_bits = bm_smem;
    u32 *s_base = bm_smem + W * wpc;
    for (int i = threadIdx.x; i < W * wpc; i += blockDim.x) s_bits[i] = colbits[i];
    for (int i = threadIdx.x; i < W; i += blockDim.x) s_base[i] = colbase[i];
    __syncthreads();
    BitmapView bm = {s_bits, s_base, H, W, wpc};
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < H * W; p += gridDim.x * blockDim.x) {
        int c = p / H, r = p - c * H;
        if (!bm_free(bm, r, c)) continue;
        int id = bm_rank(bm, r, c);
        cell_rc[id] = ((u32)r << 16) | (u32)c;
        u64 parked = 0;  // STAY on this cell parks agent i when it is agent i's goal (mapf_env.py:441-446)
        for (int i = 0; i < goals.n && i < ENT_PARK_AGENTS; ++i)
            if ((int)goals.cell[i] == id) parked |= 1ull << (ENT_PARK_SHIFT + i);
        for (int a = 0; a < 5; ++a) lut[id * 5 + a] = bm_entry(bm, r, c, a, cand_mask, pats) | (a == 0 ? parked : 0ull);
    }
}

// =====================================================================================================
// Bulk state <-> cells (state_to_locations / locations_to_state, mapf_env.py:358-371)
// =====================================================================================================
template <int WORDS>
__device__ __forceinline__ void load_state(const u64 *states, i64 b, u64 &lo, u64 &hi) {
    if (WORDS == 1) { lo = states[b]; hi = 0; }
    else { ulonglong2 v = reinterpret_cast<const ulonglong2 *>(states)[b]; lo = v.x; hi = v.y; }
}
template <int WORDS>
__device__ __forceinline__ void store_state(u64 *states, i64 b, u64 lo, u64 hi) {
    if (WORDS == 1) states[b] = lo;
    else reinterpret_cast<ulonglong2 *>(states)[b] = make_ulonglong2(lo, hi);
}

template <int N, int WORDS>
__global__ void __launch_bounds__(256) k_decode(DevSpec sp, const u64 *__restrict__ states, i64 B, int *__restrict__ cells) {
    for (i64 b = (i64)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (i64)gridDim.x * blockDim.x) {
        u64 lo, hi;
        load_state<WORDS>(states, b, lo, hi);
        int cell[N];
        decode_state<N, WORDS>(sp, lo, hi, cell);
#pragma unroll
        for (int i = 0; i < N; ++i) cells[b * N + i] = cell[i];
    }
}

template <int N, int WORDS>
__global__ void __launch_bounds__(256) k_encode(DevSpec sp, const int *__restrict__ cells, i64 B, u64 *__restrict__ states) {
    for (i64 b = (i64)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (i64)gridDim.x * blockDim.x) {
        int cell[N];
#pragma unroll
        for (int i = 0; i < N; ++i) cell[i] = min(max(cells[b * N + i], 0), sp.L - 1);
        u64 lo, hi;
        encode_state<N, WORDS>(sp, cell, lo, hi);
        store_state<WORDS>(states, b, lo, hi);
    }
}

// =====================================================================================================
// Row sources: explicit (state, action) pairs, or a slab of the full table generated from the row index
// =====================================================================================================
template <int WORDS, bool RANGE>
__device__ __forceinline__ void row_input(const DevSpec &sp, const u64 *states, const int *actions, u64 sb_lo, u64 sb_hi,
                                          i64 b, u64 &lo, u64 &hi, u32 &a) {
    if (RANGE) {
        u64 off = (u64)b / sp.nA;  // nA is a kernel-uniform constant; one 64-bit division per ROW
        a = (u32)((u64)b - off * sp.nA);
        lo = sb_lo + off;
        hi = sb_hi + (lo < sb_lo ? 1ull : 0ull);
    } else {
        load_state<WORDS>(states, b, lo, hi);
        a = (u32)actions[b];
    }
}

// len(P[s][a]) (mapf_env.py:448-479): 1 for a terminal state, else the product of merged-outcome counts
// (EXACT: the context guarantees the exact fp64-pipe divisions of the decode, i.e. its move table is staged -- here the
// table itself is still read through the read-only cache)
template <int N, int WORDS, bool RANGE, bool EXACT>
__global__ void __launch_bounds__(256) k_count(DevSpec sp, const u64 *__restrict__ states, const int *__restrict__ actions,
                                               u64 sb_lo, u64 sb_hi, i64 B, i64 *__restrict__ row_len) {
    for (i64 b = (i64)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (i64)gridDim.x * blockDim.x) {
        u64 lo, hi;
        u32 a;
        row_input<WORDS, RANGE>(sp, states, actions, sb_lo, sb_hi, b, lo, hi, a);
        int cell[N], act[N];
        decode_state<N, WORDS, EXACT>(sp, lo, hi, cell);
        decode_action<N>(a, act);
        i64 len = 1;
        if (!is_terminal<N>(sp, cell, lo, hi)) {
#pragma unroll
            for (int i = 0; i < N; ++i) len *= (i64)ENT_K(__ldg(sp.lut + cell[i] * 5 + act[i]));
        }
        row_len[b] = len;
    }
}

// =====================================================================================================
// Exclusive scan of row lengths (three small kernels; chunk = 2048 elements per block)
// =====================================================================================================
#define SCAN_CHUNK 2048
// A kernel launched with programmatic stream serialization may start before its predecessor in the stream has finished;
// everything after this wait sees the predecessor's writes.  (A no-op for an ordinary launch.)
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ i64 block_scan_256(i64 v, i64 *warp_sums, i64 &block_total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    i64 x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        i64 y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        i64 s = lane < 8 ? warp_sums[lane] : 0;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
            i64 y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        if (lane < 8) warp_sums[lane] = s;
    }
    __syncthreads();
    block_total = warp_sums[7];
    i64 incl = x + (wid > 0 ? warp_sums[wid - 1] : 0);
    __syncthreads();
    return incl - v;  // exclusive
}

static __global__ void __launch_bounds__(256) k_scan_partials(const i64 *__restrict__ in, i64 B, i64 *__restrict__ partial) {
    __shared__ i64 ws[8];
    i64 base = (i64)blockIdx.x * SCAN_CHUNK;
    i64 s = 0;
#pragma unroll
    for (int j = 0; j < SCAN_CHUNK / 256; ++j) {
        i64 i = base + j * 256 + threadIdx.x;
        s += i < B ? in[i] : 0;
    }
    i64 total;
    block_scan_256(s, ws, total);
    if (threadIdx.x == 0) partial[blockIdx.x] = total;
}

// single block: exclusive scan of the per-chunk totals in place; partial[n_chunks] = grand total.
// SPINE_THREADS threads, four consecutive totals per thread and pass (4096 per pass): the passes are serial (load ->
// barriers -> store), so their number is what this launch costs -- 2**26 one-record rows are 32768 chunks = 8 passes
// (128 passes with 256 threads and one total each took a quarter of the whole count + scan time).
#define SPINE_THREADS 1024
static __global__ void __launch_bounds__(SPINE_THREADS) k_scan_spine(i64 *partial, i64 n_chunks) {
    __shared__ i64 ws[SPINE_THREADS / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    i64 carry = 0;
    grid_dependency_wait();  // launched with programmatic stream serialization behind the kernel that writes `partial`
    for (i64 base = 0; base < n_chunks; base += 4 * SPINE_THREADS) {
        const i64 i = base + 4 * (i64)threadIdx.x;
        i64 v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = i + j < n_chunks ? partial[i + j] : 0;
        i64 x = (v[0] + v[1]) + (v[2] + v[3]);
        const i64 mine = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const i64 y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) ws[wid] = x;
        __syncthreads();
        if (wid == 0) {
            i64 t = ws[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const i64 y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += y;
            }
            ws[lane] = t;
        }
        __syncthreads();
        i64 ex = carry + (x - mine) + (wid > 0 ? ws[wid - 1] : 0);
        const i64 total = ws[SPINE_THREADS / 32 - 1];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (i + j < n_chunks) partial[i + j] = ex;
            ex += v[j];
        }
        carry += total;
        __syncthreads();  // ws is rewritten by the next pass
    }
    if (threadIdx.x == 0) partial[n_chunks] = carry;
}

// Last pass of the scan: row_ptr[i] = sum of in[0 .. i), row_ptr[B] = the total.  A thread owns two consecutive elements
// in each of four 512-element passes, so every load and store is a fully coalesced 16-byte access (vec_ok: both arrays
// 16-byte aligned).  FOLD: the chunk's offset is summed here from the raw per-chunk totals (no spine launch); otherwise
// `partial` has been scanned by k_scan_spine.
// LEN: type of the row lengths -- i64 (the public row_len arrays), or u16 / u32 for the compact lengths the fused
// count + scan keeps in its scratch when the caller does not ask for row_len (8 instead of 16 B per row between the passes).
template <bool FOLD, typename LEN>
static __global__ void __launch_bounds__(256) k_scan_final(const LEN *__restrict__ in, i64 B, const i64 *__restrict__ partial,
                                                           i64 *__restrict__ row_ptr, int vec_ok) {
    __shared__ i64 ws[8];
    const i64 base = (i64)blockIdx.x * SCAN_CHUNK;
    constexpr int PASSES = SCAN_CHUNK / 512;
    i64 v0[PASSES], v1[PASSES];
    grid_dependency_wait();  // launched with programmatic stream serialization behind the producer of `in` / `partial`
#pragma unroll
    for (int p = 0; p < PASSES; ++p) {
        const i64 i = base + p * 512 + 2 * (i64)threadIdx.x;
        if (sizeof(LEN) == 8 && vec_ok && i + 1 < B) {
            const longlong2 x = *reinterpret_cast<const longlong2 *>(in + i);
            v0[p] = x.x; v1[p] = x.y;
        } else if (sizeof(LEN) == 2 && i + 1 < B) {  // (the compact array is 4-byte aligned and i is even)
            const u32 x = *reinterpret_cast<const u32 *>(in + i);
            v0[p] = (i64)(x & 0xffffu); v1[p] = (i64)(x >> 16);
        } else if (sizeof(LEN) == 4 && i + 1 < B) {
            const uint2 x = *reinterpret_cast<const uint2 *>(in + i);
            v0[p] = (i64)x.x; v1[p] = (i64)x.y;
        } else {
            v0[p] = i < B ? (i64)in[i] : 0;
            v1[p] = i + 1 < B ? (i64)in[i + 1] : 0;
        }
    }
    i64 carry;
    if (FOLD) {
        i64 s = 0;
        for (i64 c = threadIdx.x; c < (i64)blockIdx.x; c += 256) s += partial[c];
        block_scan_256(s, ws, carry);
    } else {
        carry = partial[blockIdx.x];
    }
#pragma unroll
    for (int p = 0; p < PASSES; ++p) {
        const i64 i = base + p * 512 + 2 * (i64)threadIdx.x;
        i64 total;
        const i64 ex = block_scan_256(v0[p] + v1[p], ws, total) + carry;
        carry += total;
        if (i < B) {  // row_ptr has B + 1 entries: i + 1 <= B is always in range, and row_ptr[B] = ex + v0 when i + 1 == B
            if (vec_ok) *reinterpret_cast<longlong2 *>(row_ptr + i) = make_longlong2(ex, ex + v0[p]);
            else { row_ptr[i] = ex; row_ptr[i + 1] = ex + v0[p]; }
        }
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) row_ptr[B] = carry;
}
#define SCAN_FOLD_MAX_CHUNKS 2048  // up to this many chunks every final block sums the chunk totals before it itself (the
                                   // reads grow with the square of the chunk count: beyond ~2500 the spine launch is cheaper)

// Row lengths AND the per-chunk sums of the scan in one pass (saves the scan's first read of row_len and a launch):
// block b owns rows [b * SCAN_CHUNK, (b + 1) * SCAN_CHUNK).
template <int N, int WORDS, bool RANGE, bool EXACT, typename LEN = i64>
__global__ void __launch_bounds__(256) k_count_partials(DevSpec sp, const u64 *__restrict__ states,
                                                        const int *__restrict__ actions, u64 sb_lo, u64 sb_hi, i64 B,
                                                        LEN *__restrict__ row_len, i64 *__restrict__ partial) {
    __shared__ i64 ws[8];
    const i64 base = (i64)blockIdx.x * SCAN_CHUNK;
    u32 sum = 0;  // eight rows of at most 3**13 records
    // two halves of four rows: the four rows' inputs are loaded before the first is decoded (memory-level parallelism)
#pragma unroll
    for (int h = 0; h < SCAN_CHUNK / 256; h += 4) {
        u64 lo[4], hi[4];
        u32 a[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const i64 b = base + (h + j) * 256 + threadIdx.x;
            lo[j] = 0; hi[j] = 0; a[j] = 0;
            if (b < B) row_input<WORDS, RANGE>(sp, states, actions, sb_lo, sb_hi, b, lo[j], hi[j], a[j]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const i64 b = base + (h + j) * 256 + threadIdx.x;
            int cell[N], act[N];
            decode_state<N, WORDS, EXACT>(sp, lo[j], hi[j], cell);
            decode_action<N>(a[j], act);
            u32 len = 1;
            if (!is_terminal<N>(sp, cell, lo[j], hi[j])) {
                const u32 *hi_words = reinterpret_cast<const u32 *>(sp.lut) + 1;  // k sits in the entry's high word
#pragma unroll
                for (int i = 0; i < N; ++i) len *= (__ldg(hi_words + 2u * ((u32)cell[i] * 5u + (u32)act[i])) >> 24) & 3u;
            }
            if (b < B) {
                row_len[b] = (LEN)len;
                sum += len;
            }
        }
    }
    i64 total;
    block_scan_256((i64)sum, ws, total);
    if (threadIdx.x == 0) partial[blockIdx.x] = total;
}

// =====================================================================================================
// Expand: P[s][a] rows as CSR records (mapf_env.py:448-479)
// =====================================================================================================
// Work is partitioned by OUTPUT RECORDS, not by rows: the M = row_ptr[B] records are cut into one contiguous,
// 32-aligned range per warp, so a row of 3**13 records and a row of one record cost what they write.  A warp
//   0. finds the row holding its first record with a 32-ary search of row_ptr (one probe per lane and step),
//   A. (lane = row) decodes 32 consecutive rows: (s, a) -> cells, terminal test, the N move-table entries, row length,
//      and whether ANY pair of agents can conflict in this row at all (their destination sets touch); the row
//      descriptors go to the warp's shared-memory slab,
//   B. (lane = record) walks its record range in windows of 32 consecutive records: record w + lane belongs to lane
//      `lane`, so every store of the warp is one contiguous, fully coalesced segment.  The row of a record comes
//      from a warp-wide OR of "my row starts at position p of this window" bits (REDUX) and a popcount.
// floor(2**63 / 3**b), b = 0..13
static __constant__ u64 RECIP_POW3[14] = {
    9223372036854775808ull, 3074457345618258602ull, 1024819115206086200ull, 341606371735362066ull,
    113868790578454022ull,  37956263526151340ull,   12652087842050446ull,   4217362614016815ull,
    1405787538005605ull,    468595846001868ull,     156198615333956ull,     52066205111318ull,
    17355401703772ull,      5785133901257ull};

#define EXPAND_MAX_PAIRS 4
// chunks per warp: many agents -> rows of very different cost per record exist (pair-list overflow), spread them
#define EXPAND_CHUNKS_PER_WARP(n) ((n) >= 8 ? 4 : 1)
// smallest chunk: small batches are spread over many warps (the whole C1 table, 670 k records: 36 -> 26 us with 64 instead
// of 1024), large ones are unaffected (their share per warp is thousands of records)
#ifndef EXPAND_CHUNK_MIN
#define EXPAND_CHUNK_MIN 64
#endif
#ifndef EXPAND_LIST_MIN_AGENTS
#define EXPAND_LIST_MIN_AGENTS 8
#endif
template <int N>
struct ExpandSlab {
    u64 ent[N][32];   // move-table entry of agent i for row r
    u64 st[2][32];    // the row's own state (terminal rows re-emit it)
    u64 rcp[32];      // floor(2**63 / row length): turns a record's index within the row into a 32-bit fraction
    u32 pref[32];     // first record of row r, relative to the batch's first record
    u16 prev[N][32];  // current cell of agent i
    u32 pair[EXPAND_MAX_PAIRS][32];  // descriptors of the pairs of agents that can conflict in row r
    u8 parked[32];    // SoC: agents parked on their goal choosing STAY
    u8 flag[32];      // bit 0: terminal state; bits 1..3: number of pair descriptors; bit 4: too many, test all pairs
};

// Which pairs of agents can conflict in some outcome of a row?  A vertex conflict needs a common destination, a
// swap needs each agent's current cell among the other's destinations: both imply that the sets {current cell} +
// {merged destinations} of the two agents intersect (unused destination slots repeat slot 0).  That test rejects
// almost every pair; a pair that passes gets a descriptor
//     bits 0..4: 2i     bits 5..9: 2j     bits 10..18: conflict mask, bit 3a+b set when outcome a of agent i and
//                                                      outcome b of agent j conflict (mapf_env.py:378-389)
// so that phase B tests a record with two digit extractions and one bit test per listed pair instead of all
// N(N-1)/2 pairs.  Pairs beyond EXPAND_MAX_PAIRS switch the row to the all-pairs test.
static __device__ __noinline__ u32 pair_conflict_mask(u32 prev_i, u64 ei, u32 prev_j, u64 ej) {
    u32 mask = 0;
    for (u32 a = 0; a < 3; ++a) {
        const u32 da = (u32)(ei >> (16 * a)) & 0xffffu;
        for (u32 b = 0; b < 3; ++b) {
            const u32 db = (u32)(ej >> (16 * b)) & 0xffffu;
            const bool vertex = da == db, swap = da == prev_j && db == prev_i;
            mask |= (vertex || swap) ? 1u << (3 * a + b) : 0u;
        }
    }
    return mask;
}

template <int N>
__device__ __forceinline__ bool any_pair_can_conflict(const int (&cell)[N], const u64 (&ent)[N]) {
    bool live = false;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const u32 a0 = (u32)cell[i], a1 = (u32)ent[i] & 0xffffu, a2 = ((u32)ent[i]) >> 16, a3 = (u32)(ent[i] >> 32) & 0xffffu;
#pragma unroll
        for (int j = i + 1; j < N; ++j) {
            const u32 b0 = (u32)cell[j], b1 = (u32)ent[j] & 0xffffu, b2 = ((u32)ent[j]) >> 16,
                      b3 = (u32)(ent[j] >> 32) & 0xffffu;
            live = live || a0 == b1 || a0 == b2 || a0 == b3 || a1 == b0 || a1 == b1 || a1 == b2 || a1 == b3 ||
                   a2 == b0 || a2 == b1 || a2 == b2 || a2 == b3 || a3 == b0 || a3 == b1 || a3 == b2 || a3 == b3;
        }
    }
    return live;
}

template <int N>
__device__ __forceinline__ u32 list_conflict_pairs(const int (&cell)[N], const u64 (&ent)[N], u32 (*pair)[32], int lane) {
    u32 count = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const u32 a0 = (u32)cell[i], a1 = (u32)ent[i] & 0xffffu, a2 = ((u32)ent[i]) >> 16, a3 = (u32)(ent[i] >> 32) & 0xffffu;
#pragma unroll
        for (int j = i + 1; j < N; ++j) {
            const u32 b0 = (u32)cell[j], b1 = (u32)ent[j] & 0xffffu, b2 = ((u32)ent[j]) >> 16,
                      b3 = (u32)(ent[j] >> 32) & 0xffffu;
            const bool touch = a0 == b1 || a0 == b2 || a0 == b3 || a1 == b0 || a1 == b1 || a1 == b2 || a1 == b3 ||
                               a2 == b0 || a2 == b1 || a2 == b2 || a2 == b3 || a3 == b0 || a3 == b1 || a3 == b2 || a3 == b3;
            if (touch) {
                const u32 mask = pair_conflict_mask(a0, ent[i], b0, ent[j]);
                if (mask) {
                    if (count < EXPAND_MAX_PAIRS) pair[count][lane] = (u32)(2 * i) | ((u32)(2 * j) << 5) | (mask << 10);
                    ++count;
                }
            }
        }
    }
    return count;
}

// Phase A for one row (lane = row): decode (s, a), terminal test, the N move-table entries, the row length and its
// reciprocal, the conflict pre-filter; everything phase B needs goes to column `lane` of the warp's slab.
// Returns the row length.
template <int N, int WORDS, bool LUTS, bool RANGE>
__device__ __forceinline__ u32 expand_row_setup(const DevSpec &sp, const SmemTables &tb, ExpandSlab<N> &sl, int lane,
                                                const u64 *__restrict__ states, const int *__restrict__ actions,
                                                u64 sb_lo, u64 sb_hi, i64 b) {
    u64 slo, shi;
    u32 a;
    row_input<WORDS, RANGE>(sp, states, actions, sb_lo, sb_hi, b, slo, shi, a);
    int cell[N], act[N];
    u64 ent[N];
    decode_state<N, WORDS, LUTS>(sp, slo, shi, cell);
    decode_action<N>(a, act);
    const bool term = is_terminal<N>(sp, cell, slo, shi);
    u32 len = 1, twos = 0, threes = 0;
    // A terminal row is the single record ((1.0, False), s, 0, True) (mapf_env.py:455-456): phase B needs only the state.
    // (Safe for the register allocation only under k_expand's two-CTA launch bound: without it this early exit took 80
    // instead of 64 registers at 6 agents -- profiles/r02_ablations.txt.)
    if (term) {
        sl.st[0][lane] = slo;
        sl.st[1][lane] = shi;
        sl.flag[lane] = 1;
        return 1u;
    }
#pragma unroll
    for (int i = 0; i < N; ++i) {
        ent[i] = lut_entry<LUTS>(tb, (u32)cell[i], (u32)act[i] * 8u + (LUTS ? tb.lut : 0u));
        ent[i] = ENT_CORE(ent[i]);  // phase B reads k as e >> 56
        sl.ent[i][lane] = ent[i];
        sl.prev[i][lane] = (u16)cell[i];
        const u32 k = ENT_K(ent[i]);
        len *= k;
        twos += k == 2u ? 1u : 0u;
        threes += k == 3u ? 1u : 0u;
    }
    sl.rcp[lane] = RECIP_POW3[threes] >> twos;  // floor(floor(2**63 / 3**b) / 2**a) = floor(2**63 / (2**a 3**b))
    sl.st[0][lane] = slo;
    sl.st[1][lane] = shi;
    sl.parked[lane] = (u8)parked_agents<N>(sp, cell, act);
    // small agent counts: one bit "some pair can conflict" selects the all-pairs test (cheap for few agents);
    // from EXPAND_LIST_MIN_AGENTS agents on, the conflicting pairs are listed
    u32 n_pairs;
    if (N >= EXPAND_LIST_MIN_AGENTS) n_pairs = list_conflict_pairs<N>(cell, ent, sl.pair, lane);
    else n_pairs = any_pair_can_conflict<N>(cell, ent) ? EXPAND_MAX_PAIRS + 1u : 0u;
    sl.flag[lane] = (u8)(n_pairs <= EXPAND_MAX_PAIRS ? n_pairs << 1 : 16u);
    return len;
}

// One record of P[s][a] (mapf_env.py:448-479): `o` is its index within row `row` of the warp's slab.
struct RecordOut {
    u64 lo, hi;      // next state
    double p, reward;
    u32 flags;       // MAPF_FLAG_DONE | MAPF_FLAG_COLLISION
};

template <int N, int WORDS>
__device__ __forceinline__ RecordOut expand_record(const DevSpec &sp, const SmemTables &tb, const ExpandSlab<N> &sl,
                                                   int row, u32 flag, u32 o) {
    RecordOut out;  // the caller has dealt with terminal rows (flag bit 0)
    // Outcome digits: itertools.product, agent 0 slowest (mapf_env.py:467).  With T = row length and o the
    // record's index in the row, x = (o + 1/2) / T as a 32-bit fraction; multiplying by k_0 leaves digit 0 in
    // the integer part and the fraction of the remaining digits, and so on: ONE wide multiply per agent.
    // (T <= 3**13 < 2**21: the 2**-32 truncation of x grows to at most 2**-11 of a digit, the half-unit
    // offset keeps every digit 2**-22 away from an integer boundary.)
    u32 x = (u32)(((u64)(2u * o + 1u) * sl.rcp[row]) >> 32);
    int nxt[N];
    u32 pj[N], dv = 0;  // dv: the digits, two bits per agent
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const u64 e = sl.ent[i][row];
        const u64 wide = (u64)x * (u64)((u32)(e >> 56));  // bits 58..63 of a slab entry are zero: this is k
        const u32 d = (u32)(wide >> 32);
        x = (u32)wide;
        nxt[i] = (int)ent_dest(e, d);
        pj[i] = ENT_POFF(e) + d * 8u;
        if (N >= EXPAND_LIST_MIN_AGENTS) dv += d << (2 * i);
    }
    // probability: left-to-right product (mapf_env.py:468)
    double p = lds_f64<MAPF_SMEM_PP>(tb.base + pj[0]);
#pragma unroll
    for (int i = 1; i < N; ++i) p = __dmul_rn(p, lds_f64<MAPF_SMEM_PP>(tb.base + pj[i]));
    // reward / done / collision (mapf_env.py:225-235): clash beats goal
    bool clash = false;
    if (flag & 16u) {
        int prv[N];
#pragma unroll
        for (int i = 0; i < N; ++i) prv[i] = (int)sl.prev[i][row];
        clash = has_clash<N>(prv, nxt);
    } else if (N >= EXPAND_LIST_MIN_AGENTS) {
        for (u32 q = 0; q < (flag >> 1); ++q) {
            const u32 desc = sl.pair[q][row];
            const u32 di = (dv >> (desc & 31u)) & 3u, dj = (dv >> ((desc >> 5) & 31u)) & 3u;
            clash = clash || ((desc >> (10u + 3u * di + dj)) & 1u);
        }
    }
    encode_state<N, WORDS>(sp, nxt, out.lo, out.hi);
    const bool goal = out.lo == sp.sgoal[0] && out.hi == sp.sgoal[1];  // every agent on its goal
    const int kind = clash ? 1 : (goal ? 2 : 0);
    out.p = p;
    out.reward = lds_f64<MAPF_SMEM_REW>(tb.base + (u32)(kind * MAPF_REW_STRIDE + sl.parked[row]) * 8u);
    out.flags = (kind != 0 ? 1u : 0u) | (clash ? 2u : 0u);
    return out;
}

// From EXPAND_HEAD_MIN_AGENTS agents on, a lane caches what the first H = N - 6 agents ("head": the slowest digits of
// the product order) contribute to a record: the prefix of the probability product, their part of the next-state
// index and their digits.  The lane's records are 32 apart, the head digits change only every prod(k_i, i >= H)
// records (up to 729), so almost every record is evaluated from its six tail agents alone.
#ifndef EXPAND_HEAD_MIN_AGENTS
#define EXPAND_HEAD_MIN_AGENTS 9
#endif
#ifndef EXPAND_TAIL_AGENTS
#define EXPAND_TAIL_AGENTS 6
#endif
struct HeadCache {
    int row;      // slab row the cached values belong to (-1: none)
    u32 dvh;      // the head digits, two bits per agent
    double p;     // ((p_0 * p_1) * ...) * p_{H-1}
    u64 hpart;    // sum of dest_i * L**i over the head
};

template <int N, int WORDS>
__device__ __forceinline__ RecordOut expand_record_cached(const DevSpec &sp, const SmemTables &tb, const ExpandSlab<N> &sl,
                                                          int row, u32 flag, u32 o, HeadCache &hc) {
    constexpr int H = N - EXPAND_TAIL_AGENTS, T = EXPAND_TAIL_AGENTS;
    RecordOut out;
    u32 x = (u32)(((u64)(2u * o + 1u) * sl.rcp[row]) >> 32);
    u32 hd[H], dvh = 0;
#pragma unroll
    for (int i = 0; i < H; ++i) {  // the head digits (agent 0 slowest)
        const u64 wide = (u64)x * (u64)((u32)(sl.ent[i][row] >> 56));
        hd[i] = (u32)(wide >> 32);
        x = (u32)wide;
        dvh += hd[i] << (2 * i);
    }
    if (hc.row != row || hc.dvh != dvh) {  // a new head combination: rare
        int hcell[H];
        double p = 0.0;
#pragma unroll
        for (int i = 0; i < H; ++i) {
            const u64 e = sl.ent[i][row];
            hcell[i] = (int)ent_dest(e, hd[i]);
            const double pi = lds_f64<MAPF_SMEM_PP>(tb.base + ENT_POFF(e) + hd[i] * 8u);
            p = i == 0 ? pi : __dmul_rn(p, pi);
        }
        hc.row = row;
        hc.dvh = dvh;
        hc.p = p;
        hc.hpart = encode_word<H>(sp, hcell);
    }
    int tcell[T];
    double p = hc.p;
    u32 dv = dvh;
#pragma unroll
    for (int i = 0; i < T; ++i) {
        const u64 e = sl.ent[H + i][row];
        const u64 wide = (u64)x * (u64)((u32)(e >> 56));
        const u32 d = (u32)(wide >> 32);
        x = (u32)wide;
        tcell[i] = (int)ent_dest(e, d);
        p = __dmul_rn(p, lds_f64<MAPF_SMEM_PP>(tb.base + ENT_POFF(e) + d * 8u));  // left to right (mapf_env.py:468)
        dv += d << (2 * (H + i));
    }
    bool clash = false;
    for (u32 q = 0; q < (flag >> 1); ++q) {
        const u32 desc = sl.pair[q][row];
        const u32 di = (dv >> (desc & 31u)) & 3u, dj = (dv >> ((desc >> 5) & 31u)) & 3u;
        clash = clash || ((desc >> (10u + 3u * di + dj)) & 1u);
    }
    // next state = tail * L**H + head
    const u64 tpart = encode_word<T>(sp, tcell);
    const u64 plo = tpart * sp.powLH;
    out.lo = plo + hc.hpart;
    out.hi = WORDS == 2 ? __umul64hi(tpart, sp.powLH) + (out.lo < plo ? 1ull : 0ull) : 0ull;
    const bool goal = out.lo == sp.sgoal[0] && out.hi == sp.sgoal[1];
    const int kind = clash ? 1 : (goal ? 2 : 0);
    out.p = p;
    out.reward = lds_f64<MAPF_SMEM_REW>(tb.base + (u32)(kind * MAPF_REW_STRIDE + sl.parked[row]) * 8u);
    out.flags = (kind != 0 ? 1u : 0u) | (clash ? 2u : 0u);
    return out;
}

// dispatch: the cached evaluation needs the pair list (not the all-pairs fallback) and one-word head / tail parts
template <int N, int WORDS>
__device__ __forceinline__ RecordOut expand_record_any(const DevSpec &sp, const SmemTables &tb, const ExpandSlab<N> &sl,
                                                       int row, u32 flag, u32 o, HeadCache &hc) {
    if constexpr (N >= EXPAND_HEAD_MIN_AGENTS) {
        if (sp.head_ok && !(flag & 16u)) return expand_record_cached<N, WORDS>(sp, tb, sl, row, flag, o, hc);
    }
    return expand_record<N, WORDS>(sp, tb, sl, row, flag, o);
}

// Up to EXPAND_TWO_CTA_MAX_AGENTS agents two 512-thread CTAs fit an SM (staged table + 16 row slabs each) as long as the
// kernel stays within 64 registers: without the bound a small change in phase A (e.g. the terminal-row shortcut) lets the
// allocator take 80 and silently halves the occupancy (6 agents: 61 -> 54 % of the roofline).
// 7 agents compile to 64 registers without a spill under the bound (80 without it: 57.9 -> 63.7 % of the roofline);
// 8 and 9 agents spill under it and lose 3-6 %.
#ifndef EXPAND_TWO_CTA_MAX_AGENTS
#define EXPAND_TWO_CTA_MAX_AGENTS 7
#endif
// CTA size of k_expand (with staged tables): from EXPAND_WIDE_MIN_AGENTS agents on only one CTA fits an SM anyway (90-106
// registers), a 768-thread CTA (80 registers, some spills) brings 24 instead of 16 warps: 8 / 9 agents 51.1 / 47.1 ->
// 54.0 / 50.1 % of the roofline, 10 agents unchanged.  (The host falls back to 512 threads when the slabs of 24 warps do
// not fit next to a large staged table.)
#ifndef EXPAND_WIDE_MIN_AGENTS
#define EXPAND_WIDE_MIN_AGENTS 8
#endif
#ifndef EXPAND_WIDE_THREADS
#define EXPAND_WIDE_THREADS 768
#endif
#define EXPAND_THREADS(N) ((N) >= EXPAND_WIDE_MIN_AGENTS ? EXPAND_WIDE_THREADS : MAPF_MAX_THREADS)
template <int N, int WORDS, bool LUTS, bool RANGE>
__global__ void __launch_bounds__(EXPAND_THREADS(N), (N <= EXPAND_TWO_CTA_MAX_AGENTS ? 2 : 1))
k_expand(DevSpec sp, const u64 *__restrict__ states, const int *__restrict__ actions, u64 sb_lo, u64 sb_hi, i64 B,
         const i64 *__restrict__ row_ptr, u64 *__restrict__ next_state, double *__restrict__ prob,
         double *__restrict__ reward, u8 *__restrict__ flags) {
    extern __shared__ __align__(16) unsigned char smem[];
    SmemTables tb = tables_begin<LUTS>(sp, smem);
    const u32 FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const u32 lane_le = 0xffffffffu >> (31 - lane);
    ExpandSlab<N> &sl = reinterpret_cast<ExpandSlab<N> *>(smem + MAPF_SMEM_LUT + staged_table_bytes<LUTS>(sp))[wid];
    const i64 M = row_ptr[B];
    const i64 n_warps = (i64)gridDim.x * (blockDim.x >> 5);
    // Records are dealt out in chunks of consecutive records, chunk c to warp c mod n_warps, EXPAND_CHUNKS_PER_WARP(N)
    // chunks per warp (at least EXPAND_CHUNK_MIN records each, a multiple of 32): a row whose records are expensive
    // (more conflicting pairs than the list holds) or a giant row is spread over several warps instead of making
    // one warp the straggler of the launch, at the price of one row search per chunk.
    i64 per = (M + n_warps * EXPAND_CHUNKS_PER_WARP(N) - 1) / (n_warps * EXPAND_CHUNKS_PER_WARP(N));
    per = ((per < EXPAND_CHUNK_MIN ? EXPAND_CHUNK_MIN : per) + 31) & ~31ll;
    const i64 n_chunks = (M + per - 1) / per;
    tables_wait<LUTS>(smem);
    HeadCache hc;
    constexpr bool MULTI = EXPAND_CHUNKS_PER_WARP(N) > 1;
    for (i64 chunk = (i64)blockIdx.x * (blockDim.x >> 5) + wid; chunk < n_chunks; chunk += n_warps) {
        const i64 lo = chunk * per;
        const i64 hi = lo + per < M ? lo + per : M;
        // ---------------- 0: the row r with row_ptr[r] <= lo < row_ptr[r + 1]
        i64 r;
        {
            i64 a = 0, b = B;  // row_ptr[a] <= lo < row_ptr[b]
            while (b - a > 1) {
                const i64 step = (b - a + 31) >> 5;
                i64 p = a + (i64)(lane + 1) * step;
                p = p < b ? p : b;
                const int c = __popc(__ballot_sync(FULL, row_ptr[p] <= lo));  // probes are increasing: a prefix is true
                const i64 nb = a + (i64)(c + 1) * step;
                a += (i64)c * step;
                b = nb < b ? nb : b;
            }
            r = a;
        }
        for (;;) {
            __syncwarp();
            hc.row = -1;  // the slab is about to be rewritten
            // ---------------- phase A: rows r .. r + 31 (those that start before `hi`)
            const i64 b = r + lane;
            const i64 start = b < B ? row_ptr[b] : M;
#ifndef EXPAND_PREFETCH_ROWS
#define EXPAND_PREFETCH_ROWS 32
#endif
            if (EXPAND_PREFETCH_ROWS > 0 && b + EXPAND_PREFETCH_ROWS < B) {
                // the next batch's row starts and inputs: on their way to L2 while this batch is expanded (short rows are
                // bound by the two dependent round trips per batch: 2 agents 59.8 -> 63.2 % of the roofline)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(row_ptr + b + EXPAND_PREFETCH_ROWS));
                if (!RANGE) {
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(states + (b + EXPAND_PREFETCH_ROWS) * WORDS));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(actions + b + EXPAND_PREFETCH_ROWS));
                }
            }
            const i64 batch_begin = __shfl_sync(FULL, start, 0);
            const bool need = b < B && start < hi;
            const u32 len = need ? expand_row_setup<N, WORDS, LUTS, RANGE>(sp, tb, sl, lane, states, actions, sb_lo, sb_hi, b) : 0u;
            u32 incl = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const u32 y = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += y;
            }
            const u32 total = __shfl_sync(FULL, incl, 31);
            const int myrel = (int)(incl - len);  // first record of my row, relative to batch_begin
            sl.pref[lane] = (u32)myrel;
            __syncwarp();
            // ---------------- phase B: records [first, last) of this batch, in 32-aligned windows
            const i64 batch_end = batch_begin + total;
            const i64 first = lo > batch_begin ? lo : batch_begin;
            const i64 last = hi < batch_end ? hi : batch_end;
            const int first_rel = (int)(first - batch_begin), last_rel = (int)(last - batch_begin);
            i64 w = first & ~31ll;
            int wrel = (int)(w - batch_begin);  // may be negative in a batch's first window
            int rows_before = __popc(__ballot_sync(FULL, need && myrel < wrel));  // rows starting before the window
            for (; wrel < last_rel; wrel += 32, w += 32) {
                const bool inwin = need && myrel >= wrel && myrel < wrel + 32;
                const u32 heads = __reduce_or_sync(FULL, inwin ? 1u << (myrel - wrel) : 0u);
                const int row = rows_before + __popc(heads & lane_le) - 1;
                rows_before += __popc(heads);
                const int rel = wrel + lane;
                if (rel < first_rel || rel >= last_rel) continue;
                const i64 idx = w + lane;
                const u32 flag = sl.flag[row];
                if (flag & 1u) {  // [((1.0, False), s, 0, True)]  (mapf_env.py:455-456)
                    store_state<WORDS>(next_state, idx, sl.st[0][row], sl.st[1][row]);
                    prob[idx] = 1.0;
                    reward[idx] = 0.0;
                    flags[idx] = 1;
                    continue;
                }
                const RecordOut rec = expand_record_any<N, WORDS>(sp, tb, sl, row, flag, (u32)rel - sl.pref[row], hc);
                store_state<WORDS>(next_state, idx, rec.lo, rec.hi);
                prob[idx] = rec.p;
                reward[idx] = rec.reward;
                flags[idx] = (u8)rec.flags;
            }
            if (batch_end >= hi || r + 32 >= B) break;
            r += 32;
        }
        if (!MULTI) break;  // one chunk per warp: no outer loop for the compiler to carry state around
    }
}

// =====================================================================================================
// Bellman backup over the table without materialising it (SURVEY.md 8f, row 1)
// =====================================================================================================
//   Q[b] = 0; for ((p, collision), s2, r, done) in P[s_b][a_b]:  Q[b] += p * (r + gamma * V[s2])
// with every operation a single IEEE binary64 operation, in the row's order -- what a planner's loop over
// env.P[s][a] computes.  Rows are taken 32 at a time by a warp (phase A as in k_expand, lane = row); phase B
// evaluates the records of those rows 32 at a time, one per lane (the expensive part: outcome digits, conflict
// test, encode, the gather of V) and parks the 32 terms in shared memory; then lane i adds the terms that belong
// to row i, in order, to its own accumulator.  The rows' sums run in parallel, each one associated exactly like the
// sequential loop, and the warp stores its 32 results in one coalesced segment.  Nothing but Q is written: the
// 25 B/record of the table never exist.
template <int N>
struct BackupSlab {
    ExpandSlab<N> sl;
    double term[32];
};

template <int N, bool LUTS, bool RANGE>
__global__ void __launch_bounds__(MAPF_MAX_THREADS)
k_backup(DevSpec sp, const u64 *__restrict__ states, const int *__restrict__ actions, u64 sb_lo, i64 B,
         const double *__restrict__ V, double gamma, double *__restrict__ Q) {
    extern __shared__ __align__(16) unsigned char smem[];
    SmemTables tb = tables_begin<LUTS>(sp, smem);
    const u32 FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const u32 lane_le = 0xffffffffu >> (31 - lane);
    BackupSlab<N> &bs = reinterpret_cast<BackupSlab<N> *>(smem + MAPF_SMEM_LUT + staged_table_bytes<LUTS>(sp))[wid];
    ExpandSlab<N> &sl = bs.sl;
    const i64 n_batches = (B + 31) >> 5;
    const i64 n_warps = (i64)gridDim.x * (blockDim.x >> 5);
    tables_wait<LUTS>(smem);
    for (i64 batch = (i64)blockIdx.x * (blockDim.x >> 5) + wid; batch < n_batches; batch += n_warps) {
        const i64 b = batch * 32 + lane;
        const bool need = b < B;
        if (!RANGE && b + 32 * n_warps < B) {  // this warp's next batch of inputs (see k_expand)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(states + b + 32 * n_warps));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(actions + b + 32 * n_warps));
        }
        HeadCache hc;
        hc.row = -1;
        const u32 len = need ? expand_row_setup<N, 1, LUTS, RANGE>(sp, tb, sl, lane, states, actions, sb_lo, 0ull, b) : 0u;
        u32 incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 y = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += y;
        }
        const int total = (int)__shfl_sync(FULL, incl, 31);
        const int myrel = (int)(incl - len), myend = (int)incl;  // my row's records: [myrel, myend)
        sl.pref[lane] = (u32)myrel;
        __syncwarp();
        double mine = 0.0;  // q = 0 (Python's sum starts from the int 0)
        int rows_before = 0;
        for (int wrel = 0; wrel < total; wrel += 32) {
            const bool inwin = need && myrel >= wrel && myrel < wrel + 32;
            const u32 heads = __reduce_or_sync(FULL, inwin ? 1u << (myrel - wrel) : 0u);
            const int row = rows_before + __popc(heads & lane_le) - 1;
            rows_before += __popc(heads);
            const int rel = wrel + lane;
            if (rel < total) {
                const u32 flag = sl.flag[row];
                double term;
                if (flag & 1u) {  // the single record of a terminal state: (1.0, s, 0, True)
                    term = __dmul_rn(1.0, __dadd_rn(0.0, __dmul_rn(gamma, __ldg(V + sl.st[0][row]))));
                } else {
                    const RecordOut rec = expand_record_any<N, 1>(sp, tb, sl, row, flag, (u32)rel - sl.pref[row], hc);
                    term = __dmul_rn(rec.p, __dadd_rn(rec.reward, __dmul_rn(gamma, __ldg(V + rec.lo))));
                }
                bs.term[lane] = term;
            }
            __syncwarp();
            // lane i: the terms of row i that fall in this window, in order
            const int ja = (myrel > wrel ? myrel : wrel) - wrel, jb = (myend < wrel + 32 ? myend : wrel + 32) - wrel;
            for (int j = ja; j < jb; ++j) mine = __dadd_rn(mine, bs.term[j]);
            __syncwarp();
        }
        if (need) Q[b] = mine;
    }
}

// V[s] = max_a Q[s][a], policy[s] = the first a that attains it (np.argmax).  A warp takes 32 consecutive states
// (lanes stride over the actions of one state at a time, lane i keeps state i's result), so V and the policy are
// written in coalesced segments.
// Fused exchange step of sharded value iteration: with `peers.n > 0` the new values are written straight into EVERY
// rank's copy of the value vector (`peers.ptr[r]` are peer-mapped device pointers, NVLink stores), at the states'
// global positions `s_begin + i` -- the all-gather of the sweep happens inside this kernel, segment by segment,
// instead of as a separate collective after it.
struct PeerList {
    double *ptr[16];
    int n;
};

static __global__ void __launch_bounds__(256)
k_greedy(const double *__restrict__ Q, i64 n_states, i64 nA, double *__restrict__ V_out, int *__restrict__ policy,
         PeerList peers, i64 s_begin) {
    const int lane = threadIdx.x & 31;
    const i64 warps = (i64)gridDim.x * (blockDim.x >> 5);
    const i64 n_groups = (n_states + 31) >> 5;
    for (i64 grp = (i64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); grp < n_groups; grp += warps) {
        double keep_v = 0.0;
        int keep_a = 0;
        const i64 s0 = grp << 5;
        const int cnt = n_states - s0 < 32 ? (int)(n_states - s0) : 32;
        for (int i = 0; i < cnt; ++i) {
            const double *q = Q + (s0 + i) * nA;
            double best = 0.0;
            i64 arg = -1;
            for (i64 a = lane; a < nA; a += 32) {
                const double v = q[a];
                if (arg < 0 || v > best) { best = v; arg = a; }  // strictly greater: the first maximum stays
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                const i64 oa = __shfl_xor_sync(0xffffffffu, arg, o);
                if (oa >= 0 && (arg < 0 || ob > best || (ob == best && oa < arg))) { best = ob; arg = oa; }
            }
            if (lane == i) { keep_v = best; keep_a = (int)arg; }
        }
        if (lane < cnt) {
            if (V_out) V_out[s0 + lane] = keep_v;
            if (policy) policy[s0 + lane] = keep_a;
            for (int r = 0; r < peers.n; ++r) peers.ptr[r][s_begin + s0 + lane] = keep_v;
        }
    }
}

// =====================================================================================================
// predecessors(s) (mapf_env.py:373-376, 414-434; SURVEY.md 8f, row 2)
// =====================================================================================================
// Per agent the candidate cells are where DOWN, UP, LEFT, RIGHT, STAY lead from its cell (the reference walks the
// move backwards with the same clamp / obstacle rule), i.e. the intended destinations in the move table; equal
// cells are kept once (the reference builds a set) and the joint set is their cartesian product, emitted with
// agent 0 slowest.
template <int N>
__device__ __forceinline__ u32 pred_options(const DevSpec &sp, u32 cell, u32 (&out)[5]) {
    const int order[5] = {3, 1, 4, 2, 0};  // DOWN, UP, LEFT, RIGHT, STAY (mapf_env.py:416-420)
    u32 k = 0;
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const u32 id = (u32)__ldg(sp.lut + cell * 5u + order[j]) & 0xffffu;  // intended destination = slot 0
        bool seen = false;
#pragma unroll
        for (int q = 0; q < 5; ++q) seen = seen || (q < (int)k && out[q] == id);
        if (!seen) {
#pragma unroll
            for (int q = 0; q < 5; ++q)
                if (q == (int)k) out[q] = id;
            ++k;
        }
    }
    return k;
}

template <int N, int WORDS>
__global__ void __launch_bounds__(256) k_pred_count(DevSpec sp, const u64 *__restrict__ states, i64 B, i64 *__restrict__ row_len) {
    for (i64 b = (i64)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (i64)gridDim.x * blockDim.x) {
        u64 lo, hi;
        load_state<WORDS>(states, b, lo, hi);
        int cell[N];
        decode_state<N, WORDS>(sp, lo, hi, cell);
        i64 len = 1;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            u32 opt[5];
            len *= (i64)pred_options<N>(sp, (u32)cell[i], opt);
        }
        row_len[b] = len;
    }
}

// one warp per state: the joint combinations are dealt to the lanes, record row_ptr[b] + j holds combination j
template <int N, int WORDS>
__global__ void __launch_bounds__(256)
k_pred_emit(DevSpec sp, const u64 *__restrict__ states, i64 B, const i64 *__restrict__ row_ptr, u64 *__restrict__ pred) {
    const int lane = threadIdx.x & 31;
    const i64 warps = (i64)gridDim.x * (blockDim.x >> 5);
    for (i64 b = (i64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); b < B; b += warps) {
        u64 lo, hi;
        load_state<WORDS>(states, b, lo, hi);
        int cell[N];
        decode_state<N, WORDS>(sp, lo, hi, cell);
        u32 opt[N][5], k[N];
#pragma unroll
        for (int i = 0; i < N; ++i) k[i] = pred_options<N>(sp, (u32)cell[i], opt[i]);
        const i64 base = row_ptr[b], len = row_ptr[b + 1] - base;
        for (i64 j = lane; j < len; j += 32) {
            u64 o = (u64)j;
            int pick[N];
#pragma unroll
            for (int i = N - 1; i >= 0; --i) {  // agent 0 slowest
                const u32 d = (u32)(o % k[i]);
                o /= k[i];
                u32 c = opt[i][0];
#pragma unroll
                for (int q = 1; q < 5; ++q) c = d == (u32)q ? opt[i][q] : c;
                pick[i] = (int)c;
            }
            u64 plo, phi;
            encode_state<N, WORDS>(sp, pick, plo, phi);
            store_state<WORDS>(pred, base + j, plo, phi);
        }
    }
}

// =====================================================================================================
// A joint state as an agent subset sees it (get_local_view, utils.py:138-157; SURVEY.md 8f, row 3)
// =====================================================================================================
struct AgentList {
    int idx[16];
    int n;
    int words_out;
};

template <int N, int WORDS>
__global__ void __launch_bounds__(256)
k_project(DevSpec sp, const u64 *__restrict__ states, i64 B, AgentList sub, u64 *__restrict__ out) {
    for (i64 b = (i64)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (i64)gridDim.x * blockDim.x) {
        u64 lo, hi;
        load_state<WORDS>(states, b, lo, hi);
        int cell[N];
        decode_state<N, WORDS>(sp, lo, hi, cell);
        // little-endian radix L over the chosen agents, in the sub-env's agent order (__init__.py:70-79)
        unsigned __int128 x = 0, w = 1;
        for (int j = 0; j < sub.n; ++j) {
            int c = cell[0];
#pragma unroll
            for (int i = 1; i < N; ++i) c = sub.idx[j] == i ? cell[i] : c;
            x += (unsigned __int128)(u32)c * w;
            w *= (unsigned __int128)(u32)sp.L;
        }
        if (sub.words_out == 1) out[b] = (u64)x;
        else { out[2 * b] = (u64)x; out[2 * b + 1] = (u64)(x >> 64); }
    }
}

// =====================================================================================================
// Checksums of a record array (mod 2**64), accumulated into out8 with atomics
// =====================================================================================================
static __global__ void __launch_bounds__(256)
k_checksum(int words, i64 n, i64 index_base, const u64 *__restrict__ next_state, const double *__restrict__ prob,
           const double *__restrict__ reward, const u8 *__restrict__ flags, u64 *out8) {
    u64 acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        u64 lo = next_state[i * words], hi = words == 2 ? next_state[i * 2 + 1] : 0;
        u32 f = flags[i];
        u64 d = f & 1u, c = (f >> 1) & 1u;
        acc[0] += 1; acc[1] += c; acc[2] += d; acc[3] += lo; acc[4] += hi;
        acc[5] += (u64)__double_as_longlong(prob[i]);
        acc[6] += (u64)__double_as_longlong(reward[i]);
        acc[7] += (u64)(index_base + i + 1) * (lo + 1 + 2 * c + 4 * d);
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) atomicAdd(out8 + k, acc[k]);
    }
}

// =====================================================================================================
// Step / rollout (MapfEnv.step, mapf_env.py:237-266)
// =====================================================================================================
// Everything about one env that does not need the move table: its decoded cells, action digits and draws.
template <int N>
struct EnvIn {
    int cell[N];
    u32 actv[N];               // intended action * 8 (+ the staged move table's address): see load_actions()
    u32 w[((N + 3) / 4) * 4];  // Philox words, one per agent
    u64 lo, hi;
};

struct EnvOut {
    u64 lo, hi;
    double reward, prob;
    u32 kind;  // 0 living, 1 clash, 2 goal, 3 step from a terminal state: done = kind != 0, collision = kind == 1
    u32 rcode; // index of `reward` in the reward table: 16 * kind + parked agents (what MAPF_OPT_COMPACT stores)
};
__device__ __forceinline__ u32 out_done(const EnvOut &o) { return o.kind != 0u ? 1u : 0u; }
__device__ __forceinline__ u32 out_coll(const EnvOut &o) { return o.kind == 1u ? 1u : 0u; }

template <int N>
__device__ __forceinline__ void env_draws(const PhiloxKeys &K, u64 env, u64 step, EnvIn<N> &in) {
#pragma unroll
    for (int b = 0; b < (N + 3) / 4; ++b) {
        Philox4 x = philox_block(K, env, step, (u32)b);
#pragma unroll
        for (int q = 0; q < 4; ++q) in.w[b * 4 + q] = x.v[q];
    }
}

// One sampled joint transition.  TAPE: agent i's uniform is u[i] (a replayed reference draw) and the choice is
// `(cumsum > u).argmax()` in fp64 (mapf_env.py:255).  Otherwise the draw is the 32-bit Philox word w, u = w * 2**-32,
// and the same comparison is made on integers: cumsum_j > u  <=>  w <= T_j (the table holds ~T_j).  The host guarantees that the last
// threshold of every pattern is 2**32 - 1 (the probabilities of a pattern add up to 1), so the index is simply the
// number of thresholds below w.
// `non_terminal` (warp-uniform): the caller knows that the state is not terminal -- a rollout with auto-reset after its
// first step, when the start state is not terminal: a step that was not done leaves distinct cells that are not the
// goals, a step that was done leaves the start state -- and the duplicate / goal tests are skipped.
template <int N, int WORDS, bool LUTS, bool TAPE>
__device__ __forceinline__ EnvOut env_step(const DevSpec &sp, const SmemTables &tb, const EnvIn<N> &in,
                                           const double *__restrict__ u, u32 opts, int (&nxt)[N], bool non_terminal = false) {
    double total;
    const bool term = non_terminal ? false : is_terminal<N>(sp, in.cell, in.lo, in.hi);
    u32 ehi[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const u64 e = lut_entry<LUTS>(tb, (u32)in.cell[i], in.actv[i]);
        ehi[i] = (u32)(e >> 32);
        const u32 row = ent_row(ehi[i], tb.base);
        u32 pick;
        if (TAPE) {
            const double ui = u[i];
            const double c0 = lds_f64<MAPF_SMEM_CUM>(row), c1 = lds_f64<MAPF_SMEM_CUM + 8>(row),
                         c2 = lds_f64<MAPF_SMEM_CUM + 16>(row);
            pick = c0 > ui ? 0u : (c1 > ui ? 1u : (c2 > ui ? 2u : 0u));
        } else {
            const uint2 t = lds_u32x2<MAPF_SMEM_THR>(row);
            const u32 w = in.w[i];
            pick = count_below(w, t.x, t.y);
        }
        nxt[i] = (int)ent_dest(e, pick);
        // a terminal state's probability is 0 (mapf_env.py:240): its first factor is the 0.0 behind the tables
        const u32 paddr = (i == 0 && term) ? tb.base + (MAPF_SMEM_PZERO - MAPF_SMEM_PP) : row + pick * 8u;
        const double pi = lds_f64<MAPF_SMEM_PP>(paddr);
        total = i == 0 ? pi : __dmul_rn(total, pi);  // 1 * p0 * p1 * ... (mapf_env.py:250,257)
    }
    const bool clash = has_clash<N>(in.cell, nxt);
    EnvOut out;
    encode_state<N, WORDS>(sp, nxt, out.lo, out.hi);
    const bool goal = out.lo == sp.sgoal[0] && out.hi == sp.sgoal[1];  // every agent on its goal
    // row of the reward table: 0 living, 1 clash (beats goal, mapf_env.py:228-233), 2 goal, 3 terminal state =
    // (s, 0, True, {"prob": 0}) (mapf_env.py:238-240), a no-op that consumes no draw
    const int kind = term ? 3 : (clash ? 1 : (goal ? 2 : 0));
    // living reward: Makespan rows of the table hold the same value for every parked count
    out.rcode = (u32)(kind * MAPF_REW_STRIDE) + parked_from_entries<N>(sp, tb.act0, ehi, in.cell, in.actv);
    out.reward = lds_f64<MAPF_SMEM_REW>(tb.base + out.rcode * 8u);
    out.prob = total;
    out.kind = (u32)kind;
    if (term) {
        out.lo = in.lo; out.hi = in.hi;
#pragma unroll
        for (int i = 0; i < N; ++i) nxt[i] = in.cell[i];
    }
    if ((opts & 1u) && kind != 0) {  // MAPF_OPT_AUTO_RESET
        out.lo = sp.s0[0]; out.hi = sp.s0[1];
#pragma unroll
        for (int i = 0; i < N; ++i) nxt[i] = (int)sp.start[i];
    }
    return out;
}

__device__ __forceinline__ u32 random_action(const DevSpec &sp, const PhiloxKeys &K, u64 env, u64 step) {
    Philox4 x = philox_block(K, env, step, 15u);
    return (u32)__umul64hi(((u64)x.v[0] << 32) | x.v[1], sp.nA);
}

// EPT = envs per thread per iteration.  EPT == 2 uses 128-bit loads/stores for the 8-byte fields (and 16-bit
// stores for the two flag bytes); the launcher picks it only when B is even and every pointer is 16-byte aligned.
// B < 2**31 (the launcher splits larger batches), so every index is 32-bit and an address is one wide multiply-add.
// The inputs of the thread's next iteration are loaded before the current one is computed (software prefetch).
template <int WORDS, int EPT>
struct RawIn {
    u64 lo[EPT], hi[EPT];
    u32 a[EPT];
};

template <int WORDS, int EPT>
__device__ __forceinline__ void load_raw(const u64 *states, const int *__restrict__ actions, u32 it, RawIn<WORDS, EPT> &r) {
    if (EPT == 2 && WORDS == 1) {
        const ulonglong2 s2 = reinterpret_cast<const ulonglong2 *>(states)[it];
        const int2 a2 = reinterpret_cast<const int2 *>(actions)[it];
        r.lo[0] = s2.x; r.lo[EPT - 1] = s2.y; r.hi[0] = 0; r.hi[EPT - 1] = 0;
        r.a[0] = (u32)a2.x; r.a[EPT - 1] = (u32)a2.y;
    } else {
#pragma unroll
        for (int q = 0; q < EPT; ++q) {
            load_state<WORDS>(states, it * EPT + q, r.lo[q], r.hi[q]);
            r.a[q] = (u32)actions[it * EPT + q];
        }
    }
}

// One item (EPT consecutive envs) of k_step: decode, sample, judge, store.  `raw` / `draws` were fetched / generated one
// iteration ahead by the caller.
// COMPACT (MAPF_OPT_COMPACT): `reward` receives one code byte per env instead of the double, `done` the flag byte
// MAPF_FLAG_DONE | MAPF_FLAG_COLLISION, `coll` nothing: 18 instead of 26 result bytes per env.
// KEEP (mapf_step_host_resident): the next states are stored twice, to `next_states` (the caller's host buffer) and to
// `keep` (the envs' device-resident states, normally the array they were read from: every thread reads an item's states
// before it writes them and no other thread touches that item, so in place is safe).
template <int N, int WORDS, bool LUTS, bool TAPE, int EPT, bool COMPACT, bool KEEP>
__device__ __forceinline__ void step_item(const DevSpec &sp, const SmemTables &tb, u32 it,
                                          const RawIn<WORDS, EPT> &raw, const u32 (&draws)[EPT][((N + 3) / 4) * 4],
                                          const double *__restrict__ uniforms, u32 opts, u64 *next_states,
                                          double *__restrict__ reward, double *__restrict__ prob, u8 *__restrict__ done,
                                          u8 *__restrict__ coll, u64 *keep) {
    constexpr int NW = ((N + 3) / 4) * 4;
    EnvIn<N> in[EPT];
    const u32 b = it * EPT;
#pragma unroll
    for (int q = 0; q < EPT; ++q) {
        in[q].lo = raw.lo[q];
        in[q].hi = raw.hi[q];
        if (!TAPE) {
#pragma unroll
            for (int j = 0; j < NW; ++j) in[q].w[j] = draws[q][j];
        }
        decode_state<N, WORDS, LUTS>(sp, in[q].lo, in[q].hi, in[q].cell);
    }
    EnvOut o[EPT];
#pragma unroll
    for (int q = 0; q < EPT; ++q) {
        load_actions<N>(sp, tb, raw.a[q], in[q].actv);
        int nxt[N];
        o[q] = env_step<N, WORDS, LUTS, TAPE>(sp, tb, in[q], TAPE ? uniforms + (size_t)(b + q) * N : nullptr, opts, nxt);
    }
    if (KEEP) {
        if (EPT == 2 && WORDS == 1) reinterpret_cast<ulonglong2 *>(keep)[it] = make_ulonglong2(o[0].lo, o[EPT - 1].lo);
        else {
#pragma unroll
            for (int q = 0; q < EPT; ++q) store_state<WORDS>(keep, b + q, o[q].lo, o[q].hi);
        }
    }
    if (EPT == 2) {
        if (WORDS == 1) reinterpret_cast<ulonglong2 *>(next_states)[it] = make_ulonglong2(o[0].lo, o[EPT - 1].lo);
        else {
            store_state<WORDS>(next_states, b, o[0].lo, o[0].hi);
            store_state<WORDS>(next_states, b + 1, o[EPT - 1].lo, o[EPT - 1].hi);
        }
        reinterpret_cast<double2 *>(prob)[it] = make_double2(o[0].prob, o[EPT - 1].prob);
        const u32 sel = o[0].kind | (o[EPT - 1].kind << 4);
        if (COMPACT) {
            reinterpret_cast<u16 *>(reward)[it] = (u16)(o[0].rcode | (o[EPT - 1].rcode << 8));
            reinterpret_cast<u16 *>(done)[it] = (u16)__byte_perm(0x01010300u, 0u, sel);  // byte `kind`: done | collision << 1
        } else {
            reinterpret_cast<double2 *>(reward)[it] = make_double2(o[0].reward, o[EPT - 1].reward);
            // both flag bytes of both envs from two byte permutes: byte `kind` of 0x01010100 is done, of 0x00000100 collision
            reinterpret_cast<u16 *>(done)[it] = (u16)__byte_perm(0x01010100u, 0u, sel);
            reinterpret_cast<u16 *>(coll)[it] = (u16)__byte_perm(0x00000100u, 0u, sel);
        }
    } else {
        store_state<WORDS>(next_states, b, o[0].lo, o[0].hi);
        prob[b] = o[0].prob;
        if (COMPACT) {
            reinterpret_cast<u8 *>(reward)[b] = (u8)o[0].rcode;
            done[b] = (u8)(out_done(o[0]) | (out_coll(o[0]) << 1));
        } else {
            reward[b] = o[0].reward;
            done[b] = (u8)out_done(o[0]);
            coll[b] = (u8)out_coll(o[0]);
        }
    }
}

template <int N, int EPT>
__device__ __forceinline__ void item_draws(const PhiloxKeys &keys, u64 env0, u64 step, u32 it,
                                           u32 (&draws)[EPT][((N + 3) / 4) * 4]) {
#pragma unroll
    for (int q = 0; q < EPT; ++q) {
        EnvIn<N> tmp;
        env_draws<N>(keys, env0 + (u64)(it * EPT + q), step, tmp);
#pragma unroll
        for (int j = 0; j < ((N + 3) / 4) * 4; ++j) draws[q][j] = tmp.w[j];
    }
}

// From STEP_WIDE_MIN_AGENTS agents on (one CTA per SM: two envs per thread want ~128 registers, which leaves 16 warps
// per SM) the step kernel runs ONE env per thread in CTAs of STEP_WIDE_THREADS threads: <= 80 registers, 24 warps per SM.
// With a staged move table the EPT = 2 k_step of those agent counts is not instantiated (mapf_inst.cu).  Measured against the
// 512-thread EPT = 2 launch (profiles/r02_ablations.txt): 7 agents +1.4 / +3.0 %, 8 agents (C4) +2.8 %, 9 agents +2.3 /
// +8.6 %, 10 agents +8.9 %; 640 or 1024 threads and two envs per thread in 768-thread CTAs (a spill) are slower.
#ifndef STEP_WIDE_MIN_AGENTS
#define STEP_WIDE_MIN_AGENTS 7
#endif
#ifndef STEP_WIDE_THREADS
#define STEP_WIDE_THREADS 768
#endif
#define STEP_THREADS(N, EPT) ((N) >= STEP_WIDE_MIN_AGENTS && (EPT) == 1 ? STEP_WIDE_THREADS : MAPF_MAX_THREADS)
template <int N, int WORDS, bool LUTS, bool TAPE, int EPT, bool COMPACT = false, bool KEEP = false>
__global__ void __launch_bounds__(STEP_THREADS(N, EPT), MAPF_MIN_BLOCKS(N))
k_step(DevSpec sp, PhiloxKeys keys, const u64 *states, const int *__restrict__ actions, u32 B,
       const double *__restrict__ uniforms, u64 step, u64 env0, u32 opts, u64 *next_states,
       double *__restrict__ reward, double *__restrict__ prob, u8 *__restrict__ done, u8 *__restrict__ coll,
       u64 *keep) {
    extern __shared__ __align__(16) unsigned char smem[];
    // Programmatic dependent launch: let the next kernel of the stream start its prologue (table staging) while
    // this grid drains, and do our own prologue before waiting for the previous grid's results to be visible.
    TRACE(0);
    asm volatile("griddepcontrol.launch_dependents;");
    SmemTables tb = tables_begin<LUTS>(sp, smem);
    TRACE(1);
    const u32 n_items = B / EPT;
    const u32 stride = gridDim.x * blockDim.x;
    u32 it = blockIdx.x * blockDim.x + threadIdx.x;
    // The slip draws depend on nothing but (seed, env, step): those of the first item are generated BEFORE the wait
    // on the previous grid (they overlap its tail and the first DRAM round trip), those of every later item at the
    // end of the iteration before it.  The prefetched inputs are double-buffered (A / B) and the loop body is written
    // out twice, so that "next" becomes "current" by renaming instead of by register moves.
    constexpr int NW = ((N + 3) / 4) * 4;
    u32 draws[EPT][NW];
    if (!TAPE && it < n_items) item_draws<N, EPT>(keys, env0, step, it, draws);
    // pull this thread's input lines towards L2 while the previous grid drains (a prefetch cannot observe stale
    // data: the loads below are issued after the wait); at most MAPF_PREFETCH_ITEMS grid-stride items ahead
    for (u32 pf = it, k = 0; pf < n_items && k < MAPF_PREFETCH_ITEMS; pf += stride, ++k) {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const unsigned char *>(states) + (size_t)pf * EPT * WORDS * 8));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(actions + (size_t)pf * EPT));
    }
    TRACE(2);
    asm volatile("griddepcontrol.wait;" ::: "memory");
    TRACE(3);
    RawIn<WORDS, EPT> raw;
    if (it < n_items) load_raw<WORDS, EPT>(states, actions, it, raw);
    // the image was requested at kernel entry: wait for it here, before the loop, not inside its first iteration
    // (measured: 10.00 -> 9.91 us per 2**20-env launch)
    tables_wait<LUTS>(smem);
#ifdef MAPF_TRACE
    u32 trace_iter = 0;
#endif
    while (it < n_items) {
        const RawIn<WORDS, EPT> cur = raw;
        const u32 it_next = it + stride;
        if (it_next < n_items) load_raw<WORDS, EPT>(states, actions, it_next, raw);  // in flight during the compute below
        step_item<N, WORDS, LUTS, TAPE, EPT, COMPACT, KEEP>(sp, tb, it, cur, draws, uniforms, opts, next_states, reward, prob,
                                                            done, coll, keep);
#ifdef MAPF_TRACE
        if (trace_iter == 0) TRACE(4);
        TRACE(8 + trace_iter);
        ++trace_iter;
#endif
        if (!TAPE && it_next < n_items) item_draws<N, EPT>(keys, env0, step, it_next, draws);
        it = it_next;
    }
    TRACE(7);
}

// T steps per launch; the env's cells stay in registers between steps (no state read, no decode after the first step),
// each step's results go to slab t of the [T, B] outputs: W + 18 bytes written per env-step (+ 4 read when the actions
// are given).  EPT = 2: a thread owns two neighbouring envs and writes their results with 128-bit stores, exactly as
// k_step does; the actions of step t + 1 are loaded, and its slip draws generated, while step t is computed.
// (two envs carried in registers across steps want ~110 registers: the EPT = 2 kernel runs ONE 512-thread CTA per SM.
// Measured on 2**20 C2 envs, T = 32, actions given: 512 x 1 9.42 us per step, 256 x 2 9.85, 256 x 3 (80 registers) 10.68 --
// with 512 threads per SM every thread owns 6.92 env pairs, 98.8 % of 7 full rounds; 768 threads leave 4.61 of 5.)
#ifndef MAPF_ROLLOUT2_THREADS
#define MAPF_ROLLOUT2_THREADS 512
#endif
#ifndef MAPF_ROLLOUT2_BLOCKS
#define MAPF_ROLLOUT2_BLOCKS(N) 1
#endif
// GIVEN: the actions are an input (int32[T, B]); otherwise (actions == NULL) a uniformly random policy is drawn on the
// device -- two instantiations, so that neither carries the other's registers and code through the step loop.
template <int N, int WORDS, bool LUTS, bool TAPE, int EPT, bool GIVEN>
__global__ void __launch_bounds__((EPT == 2 ? MAPF_ROLLOUT2_THREADS : MAPF_MAX_THREADS),
                                   (EPT == 2 ? MAPF_ROLLOUT2_BLOCKS(N) : MAPF_MIN_BLOCKS(N)))
k_rollout(DevSpec sp, PhiloxKeys keys, u64 *states, const int *__restrict__ actions, i64 T, u32 B,
          const double *__restrict__ uniforms, u64 step0, u64 env0, u32 opts, u64 *__restrict__ next_states,
          double *__restrict__ reward, double *__restrict__ prob, u8 *__restrict__ done, u8 *__restrict__ coll) {
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr int NW = ((N + 3) / 4) * 4;
    SmemTables tb = tables_begin<LUTS>(sp, smem);
    const u32 n_items = B / EPT;  // the launcher picks EPT = 2 only for even B
    bool ready = false;
    for (u32 it = blockIdx.x * blockDim.x + threadIdx.x; it < n_items; it += gridDim.x * blockDim.x) {
        EnvIn<N> in[EPT];
        const u32 b = it * EPT;
        u32 a_next[EPT];
#pragma unroll
        for (int q = 0; q < EPT; ++q) {
            load_state<WORDS>(states, b + q, in[q].lo, in[q].hi);
            // the random policy's action is drawn one step ahead as well (its Philox block is off the step's critical path)
            a_next[q] = GIVEN ? (u32)actions[b + q] : random_action(sp, keys, env0 + (u64)(b + q), step0);
            if (!TAPE) env_draws<N>(keys, env0 + (u64)(b + q), step0, in[q]);
        }
#pragma unroll
        for (int q = 0; q < EPT; ++q) decode_state<N, WORDS, LUTS>(sp, in[q].lo, in[q].hi, in[q].cell);
        if (!ready) { tables_wait<LUTS>(smem); ready = true; }
        // with auto-reset every state after the first step is known not to be terminal (see env_step)
        const bool chain_non_terminal = (opts & 1u) && !sp.s0_terminal;
        size_t o = b;     // env-major position inside slab t
        size_t ov = it;   // the same in units of EPT envs
        for (i64 t = 0; t < T; ++t, o += B, ov += n_items) {
            const u64 stp = step0 + (u64)t;
            u32 a_cur[EPT];
#pragma unroll
            for (int q = 0; q < EPT; ++q) a_cur[q] = a_next[q];
            if (GIVEN && t + 1 < T) {  // in flight during the compute below
                if (EPT == 2) {
                    const int2 a2 = *reinterpret_cast<const int2 *>(actions + o + B);
                    a_next[0] = (u32)a2.x; a_next[EPT - 1] = (u32)a2.y;
                } else {
                    a_next[0] = (u32)actions[o + B];
                }
            }
            EnvOut r[EPT];
            int nxt[EPT][N];
#pragma unroll
            for (int q = 0; q < EPT; ++q) {
                load_actions<N>(sp, tb, a_cur[q], in[q].actv);
                r[q] = env_step<N, WORDS, LUTS, TAPE>(sp, tb, in[q], TAPE ? uniforms + (o + q) * N : nullptr, opts, nxt[q],
                                                      chain_non_terminal && t > 0);
            }
            if (EPT == 2) {
                if (WORDS == 1) reinterpret_cast<ulonglong2 *>(next_states)[ov] = make_ulonglong2(r[0].lo, r[EPT - 1].lo);
                else {
                    store_state<WORDS>(next_states, o, r[0].lo, r[0].hi);
                    store_state<WORDS>(next_states, o + 1, r[EPT - 1].lo, r[EPT - 1].hi);
                }
                reinterpret_cast<double2 *>(reward)[ov] = make_double2(r[0].reward, r[EPT - 1].reward);
                reinterpret_cast<double2 *>(prob)[ov] = make_double2(r[0].prob, r[EPT - 1].prob);
                const u32 sel = r[0].kind | (r[EPT - 1].kind << 4);  // see step_item()
                reinterpret_cast<u16 *>(done)[ov] = (u16)__byte_perm(0x01010100u, 0u, sel);
                reinterpret_cast<u16 *>(coll)[ov] = (u16)__byte_perm(0x00000100u, 0u, sel);
            } else {
                store_state<WORDS>(next_states, o, r[0].lo, r[0].hi);
                reward[o] = r[0].reward;
                prob[o] = r[0].prob;
                done[o] = (u8)out_done(r[0]);
                coll[o] = (u8)out_coll(r[0]);
            }
            // carry the envs forward in registers (cells of the possibly reset next state); next step's draws
#pragma unroll
            for (int q = 0; q < EPT; ++q) {
                in[q].lo = r[q].lo;
                in[q].hi = r[q].hi;
#pragma unroll
                for (int i = 0; i < N; ++i) in[q].cell[i] = nxt[q][i];
                if (!TAPE && t + 1 < T) env_draws<N>(keys, env0 + (u64)(b + q), stp + 1, in[q]);
                if (!GIVEN && t + 1 < T) a_next[q] = random_action(sp, keys, env0 + (u64)(b + q), stp + 1);
            }
        }
#pragma unroll
        for (int q = 0; q < EPT; ++q) store_state<WORDS>(states, b + q, in[q].lo, in[q].hi);
    }
    if (!ready) tables_wait<LUTS>(smem);
    (void)NW;
}

// =====================================================================================================
// Closed-loop policy evaluation: whole episodes in registers, one 13-byte record per episode
// =====================================================================================================
// Episode e (< E) starts on the start state and takes at most T steps; step t is the step of env e0 + e at step index
// step0 + t of k_step's Philox stream without auto-reset, with the action the policy picks for the current state:
//   POLICY 0 (MAPF_POLICY_RANDOM)  the uniform joint action k_rollout draws (random_action)
//   POLICY 1 (MAPF_POLICY_JOINT)   int32 policy[s], indexed by the one-word joint state
//   POLICY 2 (MAPF_POLICY_AGENTS)  u8 policy[i * L + cell of agent i]: each agent's action from its own cell
//   POLICY 3 (MAPF_POLICY_GROUPS)  int32 tables of agent groups, read through a GroupLayout (k_evaluate_groups)
// The return G = G + disc * r, disc = disc * gamma is accumulated with single binary64 operations (no FMA), and the
// episode stops at its first done.  Nothing is stored per step: ret / length / outcome of episode e are written when it
// ends (outcome = the step's kind: 1 clash, 2 goal, 3 the start state was terminal; 0 = no done within T steps).
// A lane whose episode ends takes the next episode index of the queue (`counter`, one warp-aggregated atomic per warp
// and refill), so a warp's lanes stay busy until the queue drains instead of waiting for the warp's longest episode.

// The agent groups of a MAPF_POLICY_GROUPS policy, per agent i (built by mapf_evaluate_groups).  Group g with agents
// g_0 < g_1 < ... owns L**|g| int32 entries at off[g_0]; entry sum_k cell[g_k] * L**k holds the group's joint action,
// base 5, agent g_k's digit at 5**k.
struct GroupLayout {
    u64 mul[MAPF_MAXN][MAPF_MAXN];  // [i][j]: L**(position of j in its group) when j is in i's group, else 0
    u64 off[MAPF_MAXN];             // first entry of the table of i's group
    u64 frac[MAPF_MAXN];            // ceil(2**64 / 5**(position of i + 1)): extracts i's digit (see evaluate_episodes)
    u32 amax[MAPF_MAXN];            // 5**|i's group| - 1: larger entries are clamped to it
    u32 group[MAPF_MAXN];           // group id of i
};

// The pair (i < j) a collision step is attributed to, as i | j << 4: the lexicographically smallest pair of agents in
// different groups that clashed (a vertex or a swap conflict, the two tests of has_clash), else the smallest pair.
template <int N>
__device__ __forceinline__ u32 clash_pair(const GroupLayout &gl, const int (&prev)[N], const int (&nxt)[N]) {
    u32 any = 0xffu, cross = 0xffu;
#pragma unroll
    for (int i = N - 1; i >= 0; --i)
#pragma unroll
        for (int j = N - 1; j > i; --j)
            if (nxt[i] == nxt[j] || (nxt[i] == prev[j] && nxt[j] == prev[i])) {
                any = (u32)i | (u32)j << 4;
                if (gl.group[i] != gl.group[j]) cross = any;
            }
    return cross != 0xffu ? cross : any;
}

// =====================================================================================================
// The value table of RTDP (mapf_vtable): open addressing with linear probing, keyed by the one-word joint state
// =====================================================================================================
// `capacity` (a power of two) slots; a free slot holds VT_EMPTY, which no state equals (states are < 2**63).  Entries are
// never deleted and at most capacity / 2 slots are ever occupied, so a probe sequence meets a free slot long before it
// wraps; the probe loops are still bounded by the capacity, so that a table whose keys were never cleared cannot hang.
#define VT_EMPTY 0xffffffffffffffffull
#define VT_REFUSED 0x8000000000000000ull  // bit of the count word: a store was dropped for lack of room
struct VTableView {
    const u64 *keys;
    const double *values;
    const int *actions;
    u64 mask;  // capacity - 1
};

// the splitmix64 finalizer: the home slot of a key is vt_hash(key) & mask
__device__ __forceinline__ u64 vt_hash(u64 z) {
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

// the slot holding `key`, or -1
__device__ __forceinline__ i64 vt_find(const VTableView &vt, u64 key) {
    u64 slot = vt_hash(key) & vt.mask;
    for (u64 i = 0; i <= vt.mask; ++i, slot = (slot + 1) & vt.mask) {
        const u64 k = __ldg(vt.keys + slot);
        if (k == key) return (i64)slot;
        if (k == VT_EMPTY) break;
    }
    return -1;
}

// The additive group heuristic of a one-word state: 0.0 when s is terminal, else
//     ((0.0 + V_0[l_0(s)]) + V_1[l_1(s)]) + ...      (groups in canonical order, single binary64 additions)
// where l_g(s) is group g's local state and V_g its table at gl.off of the first agent of g.  `heads`: bit i is set when
// agent i is the first agent of its group, so walking the agents in order visits the groups in canonical order.
template <int N, bool EXACT>
__device__ __forceinline__ double vt_heuristic(const DevSpec &sp, const GroupLayout &gl, const double *hv, u32 heads,
                                               u64 s) {
    int cell[N];
    decode_state<N, 1, EXACT>(sp, s, 0ull, cell);
    if (is_terminal<N>(sp, cell, s, 0ull)) return 0.0;
    double h = 0.0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        if ((heads >> i) & 1u) {
            u64 x = gl.off[i];
#pragma unroll
            for (int j = 0; j < N; ++j) x += (u64)(u32)cell[j] * gl.mul[i][j];
            h = __dadd_rn(h, __ldg(hv + x));
        }
    }
    return h;
}

// value_of(s): the stored value when s is a key of the table, else the heuristic
template <int N, bool EXACT>
__device__ __forceinline__ double vt_value(const DevSpec &sp, const GroupLayout &gl, const double *hv, u32 heads,
                                           const VTableView &vt, u64 s) {
    const i64 slot = vt_find(vt, s);
    return slot >= 0 ? __ldg(vt.values + slot) : vt_heuristic<N, EXACT>(sp, gl, hv, heads, s);
}

// The episode loop of every policy kind.  `gl` and `conflict` are used by POLICY 3 and 4 only, `vt` by POLICY 4 only.
// (The kernels' parameters carry __restrict__; passing sp and keys by value and no qualifiers here keeps k_evaluate's
// machine code as it was before this loop was shared.)
//   POLICY 4 (MAPF_POLICY_TABLE)   the action stored with the state in a value table, else the POLICY 3 group action
template <int N, int WORDS, bool LUTS, int POLICY>
__device__ __forceinline__ void evaluate_episodes(DevSpec sp, PhiloxKeys keys, const void *policy, const GroupLayout *gl,
                                                  u32 E, u32 T, double gamma, u64 step0, u64 e0, u32 *counter,
                                                  double *ret, int *length, u8 *outcome, u8 *conflict,
                                                  const VTableView *vt = nullptr) {
    extern __shared__ __align__(16) unsigned char smem[];
    SmemTables tb = tables_begin<LUTS>(sp, smem);
    const u32 n_threads = gridDim.x * blockDim.x;
    u32 e = blockIdx.x * blockDim.x + threadIdx.x;  // the first n_threads episodes are dealt out statically
    bool live = e < E;
    EnvIn<N> in;
    u32 t = 0;
    double G = 0.0, disc = 1.0;
    in.lo = sp.s0[0];
    in.hi = sp.s0[1];
#pragma unroll
    for (int i = 0; i < N; ++i) in.cell[i] = (int)sp.start[i];
    tables_wait<LUTS>(smem);
    const u32 lane = threadIdx.x & 31u;
    // every lane of a warp stays in the loop until none is live: the refill below is a warp-wide collective
    while (__any_sync(0xffffffffu, live)) {
        bool ended = false;
        if (live) {
            const u64 env = e0 + (u64)e, stp = step0 + (u64)t;
            if constexpr (POLICY == 3 || POLICY == 4) {
                bool stored = false;
                if constexpr (POLICY == 4) {
                    const i64 slot = vt_find(*vt, in.lo);
                    if (slot >= 0) {
                        stored = true;
                        load_actions<N>(sp, tb, (u32)__ldg(vt->actions + slot), in.actv);
                    }
                }
                // Each agent indexes its own group's table with its group's local state (an unrolled N x N sum whose
                // multipliers are 0 outside the group: no register array is indexed by a run-time group id) and takes
                // its digit k of the entry v < 5**13 < 2**31: with f = v * ceil(2**64 / 5**(k + 1)) mod 2**64, f / 2**64
                // is frac(v / 5**(k + 1)) + eps, eps < 2**-33, and 5 * (the top 32 bits of f, plus 1) / 2**32 has the
                // digit as its integer part (the rounding stays below 1 / 5**k).
                if (!stored) {
                    const int *tables = reinterpret_cast<const int *>(policy);
#pragma unroll
                    for (int i = 0; i < N; ++i) {
                        u64 x = gl->off[i];
#pragma unroll
                        for (int j = 0; j < N; ++j) x += (u64)(u32)in.cell[j] * gl->mul[i][j];
                        const u32 v = min((u32)__ldg(tables + x), gl->amax[i]);
                        const u32 fhi = (u32)(((u64)v * gl->frac[i]) >> 32);
                        in.actv[i] = __umulhi(fhi + 1u, 5u) * 8u + tb.act0;
                    }
                }
            } else if (POLICY == 0) {
                load_actions<N>(sp, tb, random_action(sp, keys, env, stp), in.actv);
            } else if (POLICY == 1) {
                load_actions<N>(sp, tb, (u32)__ldg(reinterpret_cast<const int *>(policy) + in.lo), in.actv);
            } else {
                const u8 *table = reinterpret_cast<const u8 *>(policy);
#pragma unroll
                for (int i = 0; i < N; ++i)  // (an out-of-range entry is clamped to LEFT, like load_actions clamps)
                    in.actv[i] = min((u32)__ldg(table + (u32)i * (u32)sp.L + (u32)in.cell[i]), 4u) * 8u + tb.act0;
            }
            env_draws<N>(keys, env, stp, in);
            int nxt[N];
            // after a step that was not done the state is not terminal (see env_step): only step 0 needs the test
            const EnvOut o = env_step<N, WORDS, LUTS, false>(sp, tb, in, nullptr, 0u, nxt, t > 0);
            if constexpr (POLICY == 3 || POLICY == 4)  // the episode ends here: its conflict byte (MAPF_NO_CONFLICT unless a clash)
                if (conflict && (o.kind != 0u || t + 1u == T))
                    conflict[e] = (u8)(o.kind == 1u ? clash_pair<N>(*gl, in.cell, nxt) : 0xffu);
            G = __dadd_rn(G, __dmul_rn(disc, o.reward));
            disc = __dmul_rn(disc, gamma);
            ++t;
            in.lo = o.lo;
            in.hi = o.hi;
#pragma unroll
            for (int i = 0; i < N; ++i) in.cell[i] = nxt[i];
            if (o.kind != 0u || t == T) {
                ret[e] = G;
                length[e] = (int)t;
                outcome[e] = (u8)o.kind;
                ended = true;
            }
        }
        const u32 fin = __ballot_sync(0xffffffffu, ended);
        if (fin) {
            u32 base = 0;
            if (lane == (u32)(__ffs(fin) - 1)) base = atomicAdd(counter, (u32)__popc(fin));
            base = __shfl_sync(0xffffffffu, base, __ffs(fin) - 1);
            if (ended) e = n_threads + base + (u32)__popc(fin & ((1u << lane) - 1u));
        }
        if (ended) {
            live = e < E;
            t = 0;
            G = 0.0;
            disc = 1.0;
            in.lo = sp.s0[0];
            in.hi = sp.s0[1];
#pragma unroll
            for (int i = 0; i < N; ++i) in.cell[i] = (int)sp.start[i];
        }
    }
}

template <int N, int WORDS, bool LUTS, int POLICY>
__global__ void __launch_bounds__(MAPF_MAX_THREADS, MAPF_MIN_BLOCKS(N))
k_evaluate(DevSpec sp, PhiloxKeys keys, const void *__restrict__ policy, u32 E, u32 T, double gamma, u64 step0, u64 e0,
           u32 *__restrict__ counter, double *__restrict__ ret, int *__restrict__ length, u8 *__restrict__ outcome) {
    evaluate_episodes<N, WORDS, LUTS, POLICY>(sp, keys, policy, nullptr, E, T, gamma, step0, e0, counter, ret, length,
                                              outcome, nullptr);
}

// MAPF_POLICY_GROUPS: `tables` holds the groups' tables; `conflict` (may be null) receives, per episode, the pair of
// its last step's clash (clash_pair) when the episode ends in a collision, else 0xff.
template <int N, int WORDS, bool LUTS>
__global__ void __launch_bounds__(MAPF_MAX_THREADS, MAPF_MIN_BLOCKS(N))
k_evaluate_groups(DevSpec sp, PhiloxKeys keys, const int *__restrict__ tables, const __grid_constant__ GroupLayout gl,
                  u32 E, u32 T, double gamma, u64 step0, u64 e0, u32 *__restrict__ counter, double *__restrict__ ret,
                  int *__restrict__ length, u8 *__restrict__ outcome, u8 *__restrict__ conflict) {
    evaluate_episodes<N, WORDS, LUTS, 3>(sp, keys, tables, &gl, E, T, gamma, step0, e0, counter, ret, length, outcome,
                                         conflict);
}

// MAPF_POLICY_TABLE (one-word states): the action stored with the state in the value table `vt`, else the group action
// of `tables` exactly as k_evaluate_groups takes it.
template <int N, bool LUTS>
__global__ void __launch_bounds__(MAPF_MAX_THREADS, MAPF_MIN_BLOCKS(N))
k_evaluate_table(DevSpec sp, PhiloxKeys keys, const int *__restrict__ tables, const __grid_constant__ GroupLayout gl,
                 const __grid_constant__ VTableView vt, u32 E, u32 T, double gamma, u64 step0, u64 e0,
                 u32 *__restrict__ counter, double *__restrict__ ret, int *__restrict__ length, u8 *__restrict__ outcome,
                 u8 *__restrict__ conflict) {
    evaluate_episodes<N, 1, LUTS, 4>(sp, keys, tables, &gl, E, T, gamma, step0, e0, counter, ret, length, outcome,
                                     conflict, &vt);
}

// =====================================================================================================
// RTDP: the Bellman update of B states over the value table, max over actions folded in
// =====================================================================================================
//   v_out[b] = max_a Q(s_b, a),  a_out[b] = the first a attaining it (np.argmax),
//   Q(s, a) = 0; for ((p, c), s2, r, done) in P[s][a]:  Q += p * (r + gamma * value_of(s2))
// with single binary64 operations in the row's order: k_backup's sum with V[s2] replaced by value_of(s2) (vt_value).
// A warp takes G = max(1, 32 / nA) consecutive input states (rcp_nA = ceil(2**32 / nA) when G > 1) and walks their G * nA (state, action) rows 32 at a time,
// rows generated from the row index; each pass is one k_backup batch (phase A, ordered per-row sums in the slab), after
// which lane j folds the Q values of state j's rows in this pass into its running (max, first argmax).  No Q buffer
// exists.  The table is only read, so a launch is a synchronous (Jacobi) update whatever the scheduling.
// (The explicit one-CTA launch bound lets ptxas use the registers it needs: with the bare thread bound it spilled at
// 1, 4, 5 and 8 agents at 32 to 64 registers.)
template <int N, bool LUTS>
__global__ void __launch_bounds__(MAPF_MAX_THREADS, 1)
k_rtdp_backup(DevSpec sp, const u64 *__restrict__ states, i64 B, const __grid_constant__ GroupLayout gl,
              const double *__restrict__ hv, u32 heads, const __grid_constant__ VTableView vt, double gamma, u32 G,
              u32 rcp_nA, double *__restrict__ v_out, int *__restrict__ a_out) {
    extern __shared__ __align__(16) unsigned char smem[];
    SmemTables tb = tables_begin<LUTS>(sp, smem);
    const u32 FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const u32 lane_le = 0xffffffffu >> (31 - lane);
    BackupSlab<N> &bs = reinterpret_cast<BackupSlab<N> *>(smem + MAPF_SMEM_LUT + staged_table_bytes<LUTS>(sp))[wid];
    ExpandSlab<N> &sl = bs.sl;
    const u32 nA = (u32)sp.nA;  // <= 5**13 < 2**31
    const i64 stride = (i64)gridDim.x * (blockDim.x >> 5) * G;
    tables_wait<LUTS>(smem);
    for (i64 s_first = ((i64)blockIdx.x * (blockDim.x >> 5) + wid) * G; s_first < B; s_first += stride) {
        const u32 n_s = B - s_first < (i64)G ? (u32)(B - s_first) : G;
        const u32 rows = n_s * nA;
        double best = 0.0;
        int arg = -1;
        for (u32 r0 = 0; r0 < rows; r0 += 32) {
            const u32 r = r0 + (u32)lane;
            const bool need = r < rows;
            const u32 js = G == 1u ? 0u : __umulhi(r, rcp_nA);  // the lane's state within the group: r / nA (r < 32)
            HeadCache hc;
            hc.row = -1;
            // the lane's (state, action) row, staged in slab words phase A does not use (the explicit-row source: no
            // 64-bit division by nA per row as the RANGE source makes)
            u64 *row_state = reinterpret_cast<u64 *>(bs.term);
            int *row_action = reinterpret_cast<int *>(sl.pref);
            if (need) {
                row_state[lane] = states[s_first + js];
                row_action[lane] = (int)(r - js * nA);
            }
            const u32 len = need ? expand_row_setup<N, 1, LUTS, false>(sp, tb, sl, lane, row_state, row_action, 0ull, 0ull,
                                                                       (i64)lane)
                                 : 0u;
            u32 incl = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const u32 y = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += y;
            }
            const int total = (int)__shfl_sync(FULL, incl, 31);
            const int myrel = (int)(incl - len), myend = (int)incl;
            sl.pref[lane] = (u32)myrel;
            __syncwarp();
            double mine = 0.0;
            int rows_before = 0;
            for (int wrel = 0; wrel < total; wrel += 32) {
                const bool inwin = need && myrel >= wrel && myrel < wrel + 32;
                const u32 starts = __reduce_or_sync(FULL, inwin ? 1u << (myrel - wrel) : 0u);
                const int row = rows_before + __popc(starts & lane_le) - 1;
                rows_before += __popc(starts);
                const int rel = wrel + lane;
                if (rel < total) {
                    const u32 flag = sl.flag[row];
                    double term;
                    if (flag & 1u) {  // the single record of a terminal state: (1.0, s, 0, True)
                        const double v = vt_value<N, false>(sp, gl, hv, heads, vt, sl.st[0][row]);
                        term = __dmul_rn(1.0, __dadd_rn(0.0, __dmul_rn(gamma, v)));
                    } else {
                        const RecordOut rec = expand_record_any<N, 1>(sp, tb, sl, row, flag, (u32)rel - sl.pref[row], hc);
                        const double v = vt_value<N, false>(sp, gl, hv, heads, vt, rec.lo);
                        term = __dmul_rn(rec.p, __dadd_rn(rec.reward, __dmul_rn(gamma, v)));
                    }
                    bs.term[lane] = term;
                }
                __syncwarp();
                const int ja = (myrel > wrel ? myrel : wrel) - wrel, jb = (myend < wrel + 32 ? myend : wrel + 32) - wrel;
                for (int j = ja; j < jb; ++j) mine = __dadd_rn(mine, bs.term[j]);
                __syncwarp();
            }
            // fold: lane j takes the Q values of its state's rows in this pass, in action order
            bs.term[lane] = mine;
            __syncwarp();
            if ((u32)lane < n_s) {
                const u32 first = (u32)lane * nA, end = first + nA;
                const u32 ja = first > r0 ? first - r0 : 0u;
                const u32 jb = end <= r0 ? 0u : (end - r0 < 32u ? end - r0 : 32u);
                for (u32 j = ja; j < jb; ++j) {
                    const double q = bs.term[j];
                    if (arg < 0 || q > best) {  // strictly greater: the first maximum stays
                        best = q;
                        arg = (int)(r0 + j - first);
                    }
                }
            }
            __syncwarp();
        }
        if ((u32)lane < n_s) {
            v_out[s_first + lane] = best;
            a_out[s_first + lane] = arg;
        }
    }
}

// Inserts or overwrites B (key, value, action) triples; the keys of one launch are distinct.  A thread that meets a free
// slot first reserves one unit of the count word (refused, with VT_REFUSED set and the triple dropped, when capacity / 2
// slots are already taken), then claims the slot with a 64-bit compare-and-swap on its key, probing on when another
// thread claimed it first.  A key stored by an earlier launch lies before any free slot of its probe sequence and is
// overwritten in place.
static __global__ void __launch_bounds__(256)
k_vtable_store(const u64 *__restrict__ states, i64 B, const double *__restrict__ v, const int *__restrict__ a,
               u64 *keys, double *values, int *actions, u64 mask, u64 *count) {
    const u64 limit = (mask + 1) >> 1;
    unsigned long long *cnt = reinterpret_cast<unsigned long long *>(count);
    for (i64 b = (i64)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (i64)gridDim.x * blockDim.x) {
        const u64 key = states[b];
        u64 slot = vt_hash(key) & mask;
        bool reserved = false;
        for (u64 i = 0; i <= mask; ++i, slot = (slot + 1) & mask) {
            u64 k = *reinterpret_cast<volatile u64 *>(keys + slot);
            if (k == VT_EMPTY) {
                if (!reserved) {
                    u64 c = *reinterpret_cast<volatile u64 *>(count);
                    while ((c & ~VT_REFUSED) < limit) {
                        const u64 prev = atomicCAS(cnt, c, c + 1);
                        if (prev == c) { reserved = true; break; }
                        c = prev;
                    }
                    if (!reserved) {
                        atomicOr(cnt, VT_REFUSED);
                        break;
                    }
                }
                k = atomicCAS(reinterpret_cast<unsigned long long *>(keys + slot), VT_EMPTY, key);
                if (k == VT_EMPTY) k = key;  // claimed
            }
            if (k == key) {
                values[slot] = v[b];
                actions[slot] = a[b];
                break;
            }
        }
    }
}

// value_of(s) and the stored action (-1 when s is not a key) of B states
template <int N>
__global__ void __launch_bounds__(256)
k_vtable_lookup(DevSpec sp, const u64 *__restrict__ states, i64 B, const __grid_constant__ GroupLayout gl,
                const double *__restrict__ hv, u32 heads, const __grid_constant__ VTableView vt,
                double *__restrict__ v_out, int *__restrict__ a_out) {
    for (i64 b = (i64)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (i64)gridDim.x * blockDim.x) {
        const u64 s = states[b];
        const i64 slot = vt_find(vt, s);
        if (slot >= 0) {
            v_out[b] = __ldg(vt.values + slot);
            a_out[b] = __ldg(vt.actions + slot);
        } else {
            v_out[b] = vt_heuristic<N, false>(sp, gl, hv, heads, s);
            a_out[b] = -1;
        }
    }
}

// =====================================================================================================
// Heterogeneous batches (SURVEY.md 8f row 4): envs of DIFFERENT specs (grid, starts/goals, rewards) in one launch
// =====================================================================================================
// The batch is a concatenation of per-spec segments (seg_begin[i] .. seg_begin[i + 1] belong to spec i).  Every CTA
// owns one contiguous, 32-aligned range of envs and walks the segments that overlap it; at a segment change it
// re-stages that spec's shared-memory image with one bulk copy (the images of all specs of a group were built for the
// same shared-memory window) and copies the spec's DevSpec behind the largest image, from where the device functions
// read it instead of the constant bank.  Same agent count, state width and per-env semantics as k_step; the Philox
// counter is the env's index in the whole batch.  As in k_step, a thread's next env is loaded, and its slip draws are
// generated, before the current one is computed.
template <int N, int WORDS, bool TAPE>
__global__ void __launch_bounds__(MAPF_MAX_THREADS, MAPF_MIN_BLOCKS(N))
k_step_group(const DevSpec *__restrict__ specs, const u32 *__restrict__ seg_begin, u32 n_specs, u32 B, u32 spec_off,
             PhiloxKeys keys, const u64 *states, const int *__restrict__ actions, const double *__restrict__ uniforms,
             u64 step, u64 env0, u32 opts, u64 *next_states, double *__restrict__ reward, double *__restrict__ prob,
             u8 *__restrict__ done, u8 *__restrict__ coll) {
    extern __shared__ __align__(16) unsigned char smem[];
    // Programmatic dependent launch, as in k_step: the next launch of the stream may begin its prologue while this grid
    // drains, and this grid stages its first spec and generates its first draws before it waits for the previous one.
    asm volatile("griddepcontrol.launch_dependents;");
    bool waited = false;
    DevSpec *ssp = reinterpret_cast<DevSpec *>(smem + spec_off);
    const u32 bar = smem_u32(smem + MAPF_SMEM_BAR);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    SmemTables tb;
    tb.base = smem_u32(smem);
    tb.lut = smem_u32(smem + MAPF_SMEM_LUT);
    tb.act0 = tb.lut;
    tb.lut_g = nullptr;
    const u32 chunks = (B + 31u) >> 5;
    const u32 r0 = min(B, (u32)((u64)chunks * blockIdx.x / gridDim.x) << 5);
    const u32 r1 = min(B, (u32)((u64)chunks * (blockIdx.x + 1) / gridDim.x) << 5);
    // the segment that holds env r0: the last i with seg_begin[i] <= r0
    u32 s = 0;
    for (u32 lo_i = 0, hi_i = n_specs; lo_i < hi_i;) {
        const u32 mid = (lo_i + hi_i + 1) >> 1;
        if (mid < n_specs && seg_begin[mid] <= r0) { lo_i = mid; s = mid; }
        else hi_i = mid - 1;
    }
    constexpr int NW = ((N + 3) / 4) * 4;
    u32 phase = 0;
    for (u32 lo = r0; lo < r1;) {
        while (seg_begin[s + 1] <= lo) ++s;  // skips empty segments
        const u32 hi = min(r1, seg_begin[s + 1]);
        {
            __syncthreads();  // every thread is done with the previous spec's tables (and sees the barrier's init)
            const u32 *src = reinterpret_cast<const u32 *>(specs + s);
            u32 *dst = reinterpret_cast<u32 *>(ssp);
            for (u32 i = threadIdx.x; i < sizeof(DevSpec) / 4; i += blockDim.x) dst[i] = src[i];
            if (threadIdx.x == 0) {
                const DevSpec &g = specs[s];
                if (tb.base != g.smem_window) __trap();  // the action table was built for another window address
                const u32 bytes = g.image_bytes;
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
                for (u32 off = 0; off < bytes;) {
                    const u32 piece = bytes - off < 32768u ? bytes - off : 32768u;
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                     smem_u32(smem + MAPF_SMEM_IMG + off)),
                                 "l"(g.image + off), "r"(piece), "r"(bar)
                                 : "memory");
                    off += piece;
                }
            }
        }
        // the first env of this thread: its inputs and draws are on their way while the image arrives
        u32 i = lo + threadIdx.x;
        u64 r_lo = 0, r_hi = 0;
        u32 r_a = 0;
        u32 draws[NW];
        if (!TAPE && i < hi) {
            EnvIn<N> tmp;
            env_draws<N>(keys, env0 + (u64)i, step, tmp);
#pragma unroll
            for (int j = 0; j < NW; ++j) draws[j] = tmp.w[j];
        }
        if (!waited) {  // the states may be the previous launch's output: no global load before this point
            asm volatile("griddepcontrol.wait;" ::: "memory");
            waited = true;
        }
        if (i < hi) {
            load_state<WORDS>(states, i, r_lo, r_hi);
            r_a = (u32)actions[i];
        }
        __syncthreads();  // the DevSpec copy is complete
        {
            u32 ok;
            do {
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                             "selp.u32 %0, 1, 0, p;\n\t}"
                             : "=r"(ok)
                             : "r"(bar), "r"(phase)
                             : "memory");
            } while (!ok);
            phase ^= 1u;
        }
        const DevSpec &sp = *ssp;
        while (i < hi) {
            EnvIn<N> in;
            in.lo = r_lo;
            in.hi = r_hi;
            const u32 a = r_a;
            if (!TAPE) {
#pragma unroll
                for (int j = 0; j < NW; ++j) in.w[j] = draws[j];
            }
            const u32 i_next = i + blockDim.x;
            if (i_next < hi) {  // in flight during the compute below
                load_state<WORDS>(states, i_next, r_lo, r_hi);
                r_a = (u32)actions[i_next];
            }
            decode_state<N, WORDS, true>(sp, in.lo, in.hi, in.cell);
            load_actions<N>(sp, tb, a, in.actv);
            int nxt[N];
            const EnvOut o = env_step<N, WORDS, true, TAPE>(sp, tb, in, TAPE ? uniforms + (size_t)i * N : nullptr, opts, nxt);
            store_state<WORDS>(next_states, i, o.lo, o.hi);
            reward[i] = o.reward;
            prob[i] = o.prob;
            done[i] = (u8)out_done(o);
            coll[i] = (u8)out_coll(o);
            if (!TAPE && i_next < hi) {
                EnvIn<N> tmp;
                env_draws<N>(keys, env0 + (u64)i_next, step, tmp);
#pragma unroll
                for (int j = 0; j < NW; ++j) draws[j] = tmp.w[j];
            }
            i = i_next;
        }
        lo = hi;
    }
}
