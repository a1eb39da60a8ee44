// mapf_device.cuh -- device-side building blocks of the joint-transition engine (sm_100a).
//
// Reference citations are file:line relative to /root/reference/gym_mapf/envs/.
#pragma once
#include <stdint.h>

typedef unsigned long long u64;
typedef long long i64;
typedef unsigned int u32;
typedef unsigned short u16;
typedef unsigned char u8;

#define MAPF_MAXN 13
#define MAPF_REW_STRIDE 16  // reward table row: parked-agent count 0..13
#define MAPF_MAX_PATTERNS 8
#define MAPF_PAT_STRIDE 24  // bytes per pattern row: 5 rows of 24 B fall on disjoint shared-memory banks (32 B rows wrap)

// Exact unsigned 64-bit division by a run-time constant d >= 1, branch-free (Granlund-Montgomery round-up method
// with the 65-bit magic; a power of two uses magic 0): q = mulhi(x, magic); q = (((x - q) >> 1) + q) >> shift.
struct FastDiv {
    u64 magic;
    u32 shift;
    u32 pad;
};
// Division by L of a two-digit chunk x < L*L: q = umulhi(x, magic) >> shift.  For almost every L (all shipped maps)
// a round-up magic exists that is exact on that range (fix == 0); otherwise a round-down magic underestimates by at
// most one and one compare fixes it (fix == 1).
struct Div32 {
    u32 magic;
    u32 shift;
    u32 fix;
    u32 pad;
};

// Move-table entry for one (cell, intended action): what `single_agent_movements` returns (mapf_env.py:163-184).
//   bits  0..15 / 16..31 / 32..47  destination cell of merged outcome 0 / 1 / 2 (unused slots repeat slot 0)
//   bits 48..55                    24 * merge pattern id: which of the candidates {intended, right-slip,
//                                  left-slip} fell on the same cell.  It is the byte offset of the pattern's row in
//                                  the per-pattern tables, whose probabilities are the candidates' added in list
//                                  order (mapf_env.py:177-179)
//   bits 56..57                    k = number of merged outcomes (1..3)
//   bits 58..62                    only on (cell, STAY) entries: bit 58 + i is set when the cell is agent i's goal
//                                  (i < 5), i.e. agent i standing here and choosing STAY is "parked" under the
//                                  sum-of-costs criterion (mapf_env.py:441-446); bit 63 is zero
#define ENT_K(e) ((u32)((e) >> 56) & 3u)
#define ENT_POFF(e) ((u32)((e) >> 48) & 0xffu)
#define ENT_PARK_AGENTS 5
#define ENT_PARK_SHIFT 58
#define ENT_CORE(e) ((e) & 0x03ffffffffffffffull)  // without the parked bits
// byte 6 of the entry (the pattern-row offset) from its high word, zero-extended: one PRMT
__device__ __forceinline__ u32 ent_poff_hi(u32 ehi) { return __byte_perm(ehi, 0u, 0x4442); }
// shared-window address of the entry's pattern row, `base + offset`, in ONE PRMT: the window address of the dynamic
// shared memory is a multiple of 256 (checked at context creation) and the offset is below 256, so the sum is the
// base with its low byte replaced
__device__ __forceinline__ u32 ent_row(u32 ehi, u32 base) { return __byte_perm(ehi, base, 0x7652); }
// destination of merged outcome j (0..2): bytes 2j, 2j+1 of the entry, zero-extended.  The upper two selector
// nibbles 0xF replicate the (always clear) sign bit of byte 7.
__device__ __forceinline__ u32 ent_dest(u64 e, u32 j) {
    u32 d;  // PTX prmt (not __byte_perm, which documents 3-bit selectors) for the sign-replicating selector nibbles
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"((u32)e), "r"((u32)(e >> 32)), "r"(0xFF10u + 0x22u * j));
    return d;
}

// Everything a hot kernel needs about one env spec; passed by value as a kernel parameter (constant bank).
struct DevSpec {
    int n;             // agents
    int L;             // free cells
    int words;         // 64-bit words per joint state (1 or 2)
    int soc;           // 1: sum-of-costs living reward (mapf_env.py:440-446)
    int s0_terminal;   // 1: the start state itself is terminal (two starts on one cell, or every start on its goal)
    int H, Wd;         // grid height / width
    int lut_smem;      // 1: the move table is staged in shared memory
    int cand_mask;     // bit j set: candidate j (intended, right, left) has probability > 0 (mapf_env.py:172)
    u32 LL;            // L*L: a joint state is decoded two agents at a time
    u32 lut_bytes;     // size of the move table, padded to 16 B
    int limbs[8];      // words==2: 32-bit limbs that can be non-zero before the k-th division by LL
    u64 nA;            // 5**n
    u64 smax[2];       // nS - 1
    FastDiv divLL;     // division by L*L
    // Exact floor divisions on the fp64 pipe (staged kernels only, see fdiv_floor()): reciprocals rounded UP and the
    // matching constants -2**52 * reciprocal, plus the negated divisors for the one-IMAD remainders
    double invLL_up, negcLL, invL_up, negcL;
    u32 negLL, negL;
    // Two-word states: s = q * D + r with D = L**KLO(n) splits the digits into a low and a high group that are then
    // decoded independently with one-word arithmetic (split_ok: D < 2**63 and L**(n - KLO) < 2**49, so that one fp64
    // estimate of q is off by at most one).  Otherwise: long division over 32-bit limbs.
    int split_ok;
    int head_ok;       // expand: the tail agents and the agents before them each fit one word (see HeadCache)
    u64 powLH;         // L**(number of head agents)
    u64 splitD;
    double invD;
    Div32 divL;        // division by L of a two-digit chunk
    u64 s0[2];         // start state
    u64 sgoal[2];      // locations_to_state(agents_goals)
    const u64 *lut;    // [L*5] move table, global memory (it lives inside `image`)
    u16 goal[16];      // goal cell per agent (mapf_env.py:158)
    u16 start[16];
    // Everything a hot CTA keeps in shared memory, laid out in global memory exactly as it sits there (see the
    // MAPF_SMEM_* layout below), so that ONE bulk asynchronous copy per CTA stages it.
    const unsigned char *image;
    u32 image_bytes;   // multiple of 16; ends after the action table when the move table is not staged
    u32 smem_window;   // shared-window address of a hot kernel's dynamic shared memory (probed at context creation;
                       // the action table holds absolute shared-window addresses)
};

// Host-side staging of the per-pattern tables (one MAPF_PAT_STRIDE-byte row per merge pattern):
struct PatternTables {
    u32 thr[MAPF_MAX_PATTERNS][6];     // ~T_j (j = 0, 1, 2), T_j = largest 32-bit draw w with cumsum_j > w * 2**-32
    double cum[MAPF_MAX_PATTERNS][3];  // np.cumsum of the merged probabilities (mapf_env.py:255)
    double pp[MAPF_MAX_PATTERNS][3];   // merged probabilities
    double zero[2];                    // 0.0: the probability factor of a step from a terminal state
    double reward[4 * MAPF_REW_STRIDE];  // [0: living, 1: clash + living, 2: goal + living, 3: terminal = 0][parked agents]
};

__device__ __forceinline__ u64 fastdiv(u64 x, const FastDiv &d) {
    const u64 q = __umul64hi(x, d.magic);
    return (((x - q) >> 1) + q) >> d.shift;
}
// chunk -> (chunk % L, chunk / L).  EXACT: the context guarantees an exact magic (Div32::fix == 0), which holds
// whenever the move table is staged in shared memory (every L below 52186 has one); the correction is compiled out.
template <bool EXACT>
__device__ __forceinline__ void divmod_L(const DevSpec &sp, u32 x, u32 &q, u32 &r) {
    q = __umulhi(x, sp.divL.magic) >> sp.divL.shift;
    r = x - q * (u32)sp.L;
    if (!EXACT && sp.divL.fix) {
        if (r >= (u32)sp.L) { r -= (u32)sp.L; q += 1; }
    }
}

// ---- joint state <-> per-agent cells: little-endian radix L, agent 0 least significant (__init__.py:50-79) ----
// The state is split into two-digit chunks (radix L*L < 2**32) with 64-bit divisions and each chunk into its two
// digits with one 32-bit multiply-high division.
// number of low digits of the two-word split for n agents: 2 * ceil(n / 4)
#define MAPF_SPLIT_KLO(n) (2 * (((n) + 3) / 4))

// floor(x / D) for an integer 0 <= x < 2**50 held as the double d = 2**52 + x (bit pattern: 0x43300000 | high word, low
// word), on the otherwise idle fp64 pipe and with no correction step:
//   t  = RU(d * inv_up - 2**52 * inv_up) = RU(x * inv_up)      one fused multiply-add, rounded up; inv_up = RU(1 / D)
//   qd = RD(t + 2**52)                     = 2**52 + floor(t)    ulp is 1 in [2**52, 2**53)
// x / D <= x * inv_up <= t < (x / D) * (1 + 2**-51), and the fraction of x / D is at most 1 - 1/D, so t stays below the
// next integer whenever x < 2**50: floor(t) = floor(x / D).  The result is again "2**52 + q", ready for the next division.
__device__ __forceinline__ double fdiv_floor(double d, double inv_up, double negc) {
    return __dadd_rd(__fma_ru(d, inv_up, negc), 4503599627370496.0);
}
__device__ __forceinline__ double u32_as_biased_double(u32 x) { return __hiloint2double(0x43300000, (int)x); }

// digits of a one-word value, two at a time: chunk = x mod L*L by one 64-bit magic division, then chunk / L
template <int N, bool EXACT>
__device__ __forceinline__ void decode_word(const DevSpec &sp, u64 x, int *cell) {
    constexpr int PAIRS = (N + 1) / 2;
    u32 chunk[PAIRS];
    double chunk_d[PAIRS];  // EXACT: 2**52 + chunk where it fell out of a division for free (else unused)
    bool have_d[PAIRS];
#pragma unroll
    for (int p = 0; p < PAIRS; ++p) have_d[p] = false;
#pragma unroll
    for (int p = 0; p < PAIRS; ++p) {
        if (p + 1 < PAIRS) {
            if (EXACT && N - 2 * p <= 4) {
                // At most four digits left and (guaranteed with EXACT, i.e. whenever the move table is staged in shared
                // memory: L <= 5632) L**4 < 2**50: quotient on the fp64 pipe, remainder with one multiply-add.  This is
                // the last division by L*L: the quotient is the top chunk.
                const double d = __hiloint2double(0x43300000 | (int)(u32)(x >> 32), (int)(u32)x);
                const double qd = fdiv_floor(d, sp.invLL_up, sp.negcLL);
                const u32 qq = (u32)__double2loint(qd);
                chunk[p] = (u32)x + qq * sp.negLL;
                chunk[p + 1] = qq;
                chunk_d[p + 1] = qd;
                have_d[p + 1] = true;
                break;
            }
            const u64 q = fastdiv(x, sp.divLL);
            chunk[p] = (u32)x - (u32)q * sp.LL;
            x = q;
        } else {
            chunk[p] = (u32)x;
        }
    }
#pragma unroll
    for (int p = 0; p < PAIRS; ++p) {
        if (2 * p + 1 < N) {
            u32 q, r;
            if (EXACT) {  // chunk < L*L < 2**25
                const double cd = have_d[p] ? chunk_d[p] : u32_as_biased_double(chunk[p]);
                q = (u32)__double2loint(fdiv_floor(cd, sp.invL_up, sp.negcL));
                r = chunk[p] + q * sp.negL;
            } else {
                divmod_L<EXACT>(sp, chunk[p], q, r);
            }
            cell[2 * p] = (int)r;
            cell[2 * p + 1] = (int)q;
        } else {
            cell[2 * p] = (int)chunk[p];
        }
    }
}

template <int N, int WORDS, bool EXACT = false>
__device__ __forceinline__ void decode_state(const DevSpec &sp, u64 lo, u64 hi, int (&cell)[N]) {
    constexpr int PAIRS = (N + 1) / 2;
    constexpr int KLO = MAPF_SPLIT_KLO(N) < N ? MAPF_SPLIT_KLO(N) : N - 1;
    u32 chunk[PAIRS];
    if constexpr (WORDS == 1) {
        decode_word<N, EXACT>(sp, lo, cell);
        cell[N - 1] = (int)min((u32)cell[N - 1], (u32)(sp.L - 1));
        return;
    }
    if constexpr (WORDS == 2 && N >= 4) if (sp.split_ok) {  // kernel-uniform
        // q = floor(s / D) from one fp64 estimate (q < 2**49: the rounded product is floor or floor + 1), fixed
        // with the sign of the remainder, whose low 64 bits are all that is needed (|r| < D < 2**63)
        const double d = __fma_rn(__ull2double_rn(hi), 18446744073709551616.0, __ull2double_rn(lo));
        u64 q = __double2ull_rn(__dmul_rn(d, sp.invD));
        i64 r = (i64)(lo - q * sp.splitD);
        if (r < 0) { r += (i64)sp.splitD; q -= 1; }
        decode_word<KLO, EXACT>(sp, (u64)r, &cell[0]);
        decode_word<(N - KLO > 0 ? N - KLO : 1), EXACT>(sp, q, &cell[KLO < N ? KLO : 0]);
        // an out-of-range state (rejected by the host API) must still give valid table indices
#pragma unroll
        for (int i = 0; i < N; ++i) cell[i] = (int)min((u32)cell[i], (u32)(sp.L - 1));
        return;
    }
    {
        // 128-bit / LL long division over 32-bit limbs; a partial dividend (rem << 32 | limb) fits 64 bits
        u32 limb[4] = {(u32)lo, (u32)(lo >> 32), (u32)hi, (u32)(hi >> 32)};
#pragma unroll
        for (int p = 0; p < PAIRS; ++p) {
            if (p + 1 < PAIRS) {
                u64 rem = 0;
                const int nl = sp.limbs[p < 8 ? p : 7];
#pragma unroll
                for (int w = 3; w >= 0; --w) {
                    if (w < nl) {
                        const u64 cur = (rem << 32) | limb[w];
                        const u64 q = fastdiv(cur, sp.divLL);
                        rem = cur - q * sp.LL;
                        limb[w] = (u32)q;
                    }
                }
                chunk[p] = (u32)rem;
            } else {
                chunk[p] = limb[0];
            }
        }
    }
#pragma unroll
    for (int p = 0; p < PAIRS; ++p) {
        if (2 * p + 1 < N) {
            u32 q, r;
            divmod_L<EXACT>(sp, chunk[p], q, r);
            cell[2 * p] = (int)r;
            cell[2 * p + 1] = (int)q;
        } else {
            cell[2 * p] = (int)chunk[p];
        }
    }
    // an out-of-range state (rejected by the host API) can only corrupt the top digit: keep it a valid table index
    cell[N - 1] = (int)min((u32)cell[N - 1], (u32)(sp.L - 1));
}

// Horner over two-digit chunks in one word
template <int N>
__device__ __forceinline__ u64 encode_word(const DevSpec &sp, const int *cell) {
    constexpr int PAIRS = (N + 1) / 2;
    const u32 L = (u32)sp.L;
    u64 acc = 0;
#pragma unroll
    for (int p = PAIRS - 1; p >= 0; --p) {
        const u32 chunk = (2 * p + 1 < N) ? (u32)cell[2 * p + 1] * L + (u32)cell[2 * p] : (u32)cell[2 * p];
        acc = acc * sp.LL + chunk;
    }
    return acc;
}

template <int N, int WORDS>
__device__ __forceinline__ void encode_state(const DevSpec &sp, const int (&cell)[N], u64 &lo, u64 &hi) {
    constexpr int PAIRS = (N + 1) / 2;
    constexpr int KLO = MAPF_SPLIT_KLO(N) < N ? MAPF_SPLIT_KLO(N) : N - 1;
    if constexpr (WORDS == 1) {
        lo = encode_word<N>(sp, &cell[0]);
        hi = 0;
        return;
    }
    if constexpr (WORDS == 2 && N >= 4) if (sp.split_ok) {  // kernel-uniform: low and high digit groups in one word each
        const u64 vlo = encode_word<KLO>(sp, &cell[0]);
        const u64 vhi = encode_word<(N - KLO > 0 ? N - KLO : 1)>(sp, &cell[KLO < N ? KLO : 0]);
        const u64 plo = vhi * sp.splitD;
        lo = plo + vlo;
        hi = __umul64hi(vhi, sp.splitD) + (lo < plo ? 1ull : 0ull);
        return;
    }
    const u32 L = (u32)sp.L;
    u64 alo = 0, ahi = 0;
#pragma unroll
    for (int p = PAIRS - 1; p >= 0; --p) {
        const u32 chunk = (2 * p + 1 < N) ? (u32)cell[2 * p + 1] * L + (u32)cell[2 * p] : (u32)cell[2 * p];
        const u64 carry = __umul64hi(alo, (u64)sp.LL);
        ahi = ahi * sp.LL + carry;
        alo = alo * sp.LL;
        const u64 t = alo + chunk;
        ahi += (t < alo) ? 1ull : 0ull;
        alo = t;
    }
    lo = alo;
    hi = ahi;
}

template <int N>
__device__ __forceinline__ void decode_action(u32 a, int (&act)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
        u32 q = a / 5u;
        act[i] = (int)(a - q * 5u);
        a = q;
    }
}

// is_terminal (mapf_env.py:210-223): two agents on one cell, or every agent on its own goal (the state IS the goal
// state: one 64/128-bit compare instead of one compare per agent)
template <int N>
__device__ __forceinline__ bool is_terminal(const DevSpec &sp, const int (&cell)[N], u64 lo, u64 hi) {
    bool dup = false;  // (`||`: measured faster than a branch-free `|` chain, r02 ablations)
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = i + 1; j < N; ++j) dup = dup || (cell[i] == cell[j]);
    return dup || (lo == sp.sgoal[0] && hi == sp.sgoal[1]);
}

// _is_collision_transition_from_local_states (mapf_env.py:378-389): swap or vertex conflict over all pairs.
// Cells are 16-bit, so agent i's move is packed as prev | next << 16; agent j swaps with i exactly when
// next_j | prev_j << 16 equals that word.
template <int N>
__device__ __forceinline__ bool has_clash(const int (&prev)[N], const int (&nxt)[N]) {
    u32 fw[N], bw[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        fw[i] = __byte_perm((u32)prev[i], (u32)nxt[i], 0x5410);
        bw[i] = __byte_perm((u32)nxt[i], (u32)prev[i], 0x5410);
    }
    bool c = false;
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = i + 1; j < N; ++j) c = c || (nxt[i] == nxt[j]) || (fw[i] == bw[j]);
    return c;
}

// number of agents parked on their goal that chose STAY (mapf_env.py:441-446); 0 under Makespan.
// (prev ^ goal) | act is zero exactly for such an agent.
template <int N>
__device__ __forceinline__ int parked_agents(const DevSpec &sp, const int (&prev)[N], const int (&act)[N]) {
    int k = 0;
    if (sp.soc) {
#pragma unroll
        for (int i = 0; i < N; ++i) k += ((((u32)prev[i] ^ (u32)sp.goal[i]) | (u32)act[i]) == 0u) ? 1 : 0;
    }
    return k;
}

// The same count from the move-table entries of the agents' (cell, intended action): the first ENT_PARK_AGENTS
// agents carry a "parked" bit in their entry, the others are compared.  `actv` holds action * 8 + act0.
template <int N>
__device__ __forceinline__ u32 parked_from_entries(const DevSpec &sp, u32 act0, const u32 (&ehi)[N], const int (&prev)[N],
                                                   const u32 (&actv)[N]) {
    if (!sp.soc) return 0u;  // kernel-uniform: under Makespan every row of the reward table holds one value
    u32 bits = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        if (i < ENT_PARK_AGENTS) bits |= ehi[i] & (1u << (ENT_PARK_SHIFT - 32 + i));
    }
    u32 k = __popc(bits);
#pragma unroll
    for (int i = ENT_PARK_AGENTS; i < N; ++i) k += ((((u32)prev[i] ^ (u32)sp.goal[i]) | (actv[i] ^ act0)) == 0u) ? 1u : 0u;
    return k;
}

// (w > a) + (w > b) from the carry flag: w > a  <=>  w + ~a carries out of 32 bits.  The thresholds are stored
// complemented (na = ~a, nb = ~b) so each comparison is one carry-generating add.
__device__ __forceinline__ u32 count_below(u32 w, u32 na, u32 nb) {
    u32 t, n;
    asm("{\n\t.reg .u32 t0;\n\tadd.cc.u32 t0, %1, %2;\n\taddc.u32 %0, 0, 0;\n\t}" : "=r"(t) : "r"(w), "r"(na));
    asm("{\n\t.reg .u32 t0;\n\tadd.cc.u32 t0, %1, %2;\n\taddc.u32 %0, %3, 0;\n\t}" : "=r"(n) : "r"(w), "r"(nb), "r"(t));
    return n;
}

// ---- Philox4x32-10 (Salmon et al., SC'11), the counter-based generator of the device-side sampling mode -------
struct Philox4 {
    u32 v[4];
};
// The ten round keys (key + r * Weyl constants) are computed on the host once per launch and passed as a kernel
// parameter, so each round is two wide multiplies and two three-input XORs with constant-bank operands.
struct PhiloxKeys {
    u32 k[20];
};
__device__ __forceinline__ Philox4 philox4x32_10(u32 c0, u32 c1, u32 c2, u32 c3, const PhiloxKeys &K) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        // one wide multiply per product (measured faster than separate hi/lo multiplies)
        u64 p0, p1;
        asm("mul.wide.u32 %0, %1, %2;" : "=l"(p0) : "r"(c0), "r"(0xD2511F53u));
        asm("mul.wide.u32 %0, %1, %2;" : "=l"(p1) : "r"(c2), "r"(0xCD9E8D57u));
        const u32 hi0 = (u32)(p0 >> 32), lo0 = (u32)p0, hi1 = (u32)(p1 >> 32), lo1 = (u32)p1;
        const u32 n0 = hi1 ^ c1 ^ K.k[2 * r], n2 = hi0 ^ c3 ^ K.k[2 * r + 1];
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    }
    Philox4 out;
    out.v[0] = c0; out.v[1] = c1; out.v[2] = c2; out.v[3] = c3;
    return out;
}

// Counter layout of the sampling stream: (env low, env high, step low, step high<<8 | block); key = seed.
// block b < 8 supplies the slip draws of agents 4b..4b+3 (one 32-bit word w each, u = w * 2**-32);
// block 15 supplies the random-policy action (words 0,1 as a 64-bit fraction of nA).
__device__ __forceinline__ Philox4 philox_block(const PhiloxKeys &K, u64 env, u64 step, u32 block) {
    return philox4x32_10((u32)env, (u32)(env >> 32), (u32)step, ((u32)(step >> 32) << 8) | block, K);
}

// ---- shared memory: small per-pattern tables + the move table ------------------------------------------------
// Layout of the dynamic shared memory of every hot kernel (pattern tables have one 32-byte row per pattern):
//   [0, 16)        mbarrier of the bulk copy
//   [16, 208)      thr    u32[8][6]
//   [208, 400)     cum    f64[8][3]
//   [400, 592)     pp     f64[8][3]
//   [592, 608)     0.0
//   [608, 1120)    reward f64[64]: rows living, clash + living, goal + living, terminal state (zeros)
//   [1120, 6128)   action table u16[625][4]: for a joint action of four agents (base-5 digits, agent 0 least
//                  significant, __init__.py:26) the byte offsets action * 8 of their move-table entries, plus the
//                  table's shared-window address when it is staged -- one 8-byte load per four agents replaces the
//                  divisions by 5
//   [6128 ...)     move table u64[L*5] (when staged), then kernel-specific scratch
// Bytes [16, ...) are a verbatim copy of DevSpec::image.
#define MAPF_SMEM_BAR 0
#define MAPF_SMEM_IMG 16
#define MAPF_SMEM_THR 16
#define MAPF_SMEM_CUM 208
#define MAPF_SMEM_PP 400
#define MAPF_SMEM_PZERO 592
#define MAPF_SMEM_REW 608
#define MAPF_SMEM_ACT 1120
#define MAPF_SMEM_LUT 6128

// Shared memory is addressed through 32-bit shared-window addresses and explicit ld.shared, so that every table
// access is one LDS with an immediate offset (no generic-address arithmetic).
struct SmemTables {
    u32 base;          // shared-window address of the dynamic shared memory
    u32 lut;           // shared-window address of the staged move table
    u32 act0;          // what the action table holds for STAY: the staged table's address, or 0
    const u64 *lut_g;  // the move table in global memory
};

__device__ __forceinline__ u32 smem_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }

template <int OFF>
__device__ __forceinline__ u64 lds_u64(u32 addr) {
    u64 v;
    asm volatile("ld.shared.u64 %0, [%1+%2];" : "=l"(v) : "r"(addr), "n"(OFF));
    return v;
}
template <int OFF>
__device__ __forceinline__ double lds_f64(u32 addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1+%2];" : "=d"(v) : "r"(addr), "n"(OFF));
    return v;
}
template <int OFF>
__device__ __forceinline__ uint2 lds_u32x2(u32 addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2+%3];" : "=r"(v.x), "=r"(v.y) : "r"(addr), "n"(OFF));
    return v;
}

// Start staging: ONE thread issues the bulk asynchronous copy (cp.async.bulk, the TMA engine) of the whole image;
// it completes on an mbarrier.  Compute that does not need the tables (global loads, state decode, Philox) overlaps
// with it.  Call tables_wait() before the first table access.
template <bool LUTS>
__device__ __forceinline__ SmemTables tables_begin(const DevSpec &sp, unsigned char *smem) {
    const u32 bar = smem_u32(smem + MAPF_SMEM_BAR);
    if (threadIdx.x == 0) {
        if (smem_u32(smem) != sp.smem_window) __trap();  // the action table was built for another window address
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const u32 bytes = sp.image_bytes;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        u32 off = 0;
        while (off < bytes) {  // pieces of at most 32 KiB
            const u32 piece = bytes - off < 32768u ? bytes - off : 32768u;
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             smem_u32(smem + MAPF_SMEM_IMG + off)),
                         "l"(sp.image + off), "r"(piece), "r"(bar)
                         : "memory");
            off += piece;
        }
    }
    __syncthreads();  // the initialised barrier is visible to every thread before it polls
    SmemTables t;
    t.base = smem_u32(smem);
    t.lut = smem_u32(smem + MAPF_SMEM_LUT);
    t.act0 = LUTS ? t.lut : 0u;
    asm volatile("" : "+r"(t.base), "+r"(t.lut));  // opaque: keep both in registers instead of re-deriving them
    t.lut_g = sp.lut;
    return t;
}

template <bool LUTS>
__device__ __forceinline__ void tables_wait(unsigned char *smem) {
    const u32 bar = smem_u32(smem + MAPF_SMEM_BAR);
    u32 ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok)
                     : "r"(bar), "r"(0u)
                     : "memory");
    } while (!ok);
}

template <int OFF>
__device__ __forceinline__ u32 lds_u16(u32 addr) {
    u32 v;
    asm volatile("ld.shared.u16 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF));
    return v;
}

// Joint action -> per agent `action * 8 (+ the staged move table's address)`, straight from the action table.
template <int N>
__device__ __forceinline__ void load_actions(const DevSpec &sp, const SmemTables &tb, u32 a, u32 (&actv)[N]) {
    a = min(a, (u32)sp.nA - 1u);  // an invalid action (rejected by the host API) must not index outside the table
#pragma unroll
    for (int c = 0; c < (N + 3) / 4; ++c) {
        u32 idx = a;
        if (c + 1 < (N + 3) / 4) {
            const u32 q = __umulhi(a, 0x68DB8BADu) >> 8;  // a / 625, exact for a < 2**31 (nA <= 5**13)
            idx = a - q * 625u;
            a = q;
        }
        const uint2 v = lds_u32x2<MAPF_SMEM_ACT>(tb.base + idx * 8u);  // ONE load: four 16-bit values
        if (4 * c + 0 < N) actv[4 * c + 0] = v.x & 0xffffu;
        if (4 * c + 1 < N) actv[4 * c + 1] = v.x >> 16;
        if (4 * c + 2 < N) actv[4 * c + 2] = v.y & 0xffffu;
        if (4 * c + 3 < N) actv[4 * c + 3] = v.y >> 16;
    }
}

// bytes of shared memory the staged table occupies behind MAPF_SMEM_LUT (kernel scratch follows it)
template <bool LUTS>
__device__ __forceinline__ u32 staged_table_bytes(const DevSpec &sp) {
    return LUTS ? sp.lut_bytes : 0u;
}

// move-table entry of (cell, action): `act8` is action * 8 (+ the table's shared-window address when staged)
template <bool LUTS>
__device__ __forceinline__ u64 lut_entry(const SmemTables &tb, u32 cell, u32 act8) {
    if (LUTS) return lds_u64<0>(cell * 40u + act8);
    return __ldg(reinterpret_cast<const u64 *>(reinterpret_cast<const unsigned char *>(tb.lut_g) + (cell * 40u + act8)));
}
