/* mapf_b200.h -- C ABI of the B200 joint-transition engine for gym-mapf.
 *
 * The reference (LevyvoNet/gym-mapf) is pure Python and has no FFI: its boundary for this path is the Python
 * API of `MapfEnv` (gym_mapf/envs/mapf_env.py).  Each entry point below states the reference interface it
 * replaces as file:line relative to /root/reference/gym_mapf/envs/.  The Python package `gym_mapf_b200`
 * (gym_mapf_b200/) binds this library with ctypes (gym_mapf_b200/_native.py); INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *  - Plain C symbols, no C++ types or exceptions cross the boundary.
 *  - Every function returns MAPF_OK (0) or a negative mapf_status; mapf_last_error() returns the message of the
 *    last failure on the calling thread.
 *  - Unless a parameter is documented as HOST memory, data pointers are caller-owned DEVICE pointers (for
 *    example a torch tensor's data_ptr()); the library never frees or retains them.
 *  - Calls taking a `stream` are asynchronous on that CUDA stream (pass 0 for the legacy default stream, or
 *    torch.cuda.current_stream().cuda_stream); they do not synchronise and do not allocate.
 *  - A context is immutable after creation and may be shared by host threads; one context per device.
 *  - Joint states are little-endian mixed-radix integers with agent 0 least significant (envs/__init__.py:70-79).
 *    A state occupies `state_words` 64-bit words (mapf_info): 1 when L**n < 2**63, else 2 (low word first).
 *    With torch these are int64[B] and int64[B,2].
 *  - Joint actions are int32 base-5 integers, agent 0 least significant, digit order STAY, UP, RIGHT, DOWN, LEFT
 *    (envs/__init__.py:26, mapf_env.py:97-102).
 *  - "cells" are per-agent local state ids: the rank of a free cell in column-major order (grid.py:37-40,
 *    mapf_env.py:142-143).
 *  - Rewards and probabilities are IEEE binary64, computed in the reference's operation order (bit-exact).
 */
#ifndef MAPF_B200_H
#define MAPF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MAPF_MAX_AGENTS 13 /* 5**13 < 2**31: joint actions stay int32 */
#define MAPF_MAX_CELLS 65535 /* cell ids are 16-bit inside the move table (largest shipped map: 47 540) */

typedef enum mapf_status {
    MAPF_OK = 0,
    MAPF_ERR_INVALID = -1,     /* bad argument (NULL, negative size, ...) */
    MAPF_ERR_KEY = -2,         /* start/goal on an obstacle or off the grid: the reference's KeyError (mapf_env.py:369) */
    MAPF_ERR_UNSUPPORTED = -3, /* more than MAPF_MAX_AGENTS agents, more than MAPF_MAX_CELLS cells, L**n >= 2**127 */
    MAPF_ERR_CUDA = -4,        /* a CUDA call failed; the text is in mapf_last_error() */
    MAPF_ERR_NO_DEVICE = -5    /* no usable CUDA device: there is no CPU fallback */
} mapf_status;

enum { MAPF_SOC = 0, MAPF_MAKESPAN = 1 }; /* mapf_env.py:31-33 OptimizationCriteria */

/* flag bits of a transition record */
enum { MAPF_FLAG_DONE = 1, MAPF_FLAG_COLLISION = 2, MAPF_FLAG_TERMINAL = 4 };

/* step / rollout option bits */
enum {
    MAPF_OPT_AUTO_RESET = 1, /* an env whose step returned done is put back on the start state (next_state holds
                                the start state for it); off = the reference's semantics (mapf_env.py:237-266) */
    MAPF_OPT_COMPACT = 4,    /* mapf_step / mapf_step_host: 18 instead of 26 result bytes per env (the host link is the bound
                                of the end-to-end step).  `reward` then receives ONE BYTE per env, a code into the 64 doubles
                                of mapf_ctx_reward_table (every reward the env can return, computed in the reference's order:
                                mapf_env.py:225-235, 436-446), and `done` one byte with MAPF_FLAG_DONE | MAPF_FLAG_COLLISION;
                                `collision` is not written (may be NULL).  next_states and prob are unchanged. */
    MAPF_OPT_SHARE_SM = 2    /* mapf_step only: launch ONE resident CTA per SM instead of filling the GPU.  For callers
                                that keep their envs in two independent pools and step each pool on its own stream
                                (every pool is a chain of dependent launches, mapf_env.py:237-266 called once per env
                                and step): the two chains then share every SM, and the drain / fill of one pool's
                                launch boundary is covered by the other pool's compute.  Results are identical. */
};

/* Everything MapfEnv.__init__ receives (mapf_env.py:116-125); all HOST memory, copied by mapf_ctx_create. */
typedef struct mapf_spec {
    int32_t height, width;
    const uint8_t *obstacles; /* row-major height*width bytes, non-zero = obstacle '@' (grid.py:9-25) */
    int32_t n_agents;
    const int32_t *start_rc;  /* 2*n_agents ints: (row, col) per agent (mapf_env.py:128) */
    const int32_t *goal_rc;   /* 2*n_agents ints */
    double fail_prob;         /* right/left slip = fail_prob / 2 each (mapf_env.py:131-132) */
    double reward_of_clash, reward_of_goal, reward_of_living;
    int32_t criterion;        /* MAPF_SOC or MAPF_MAKESPAN */
} mapf_spec;

typedef struct mapf_info {
    int32_t n_agents;
    int32_t n_cells;         /* L = len(valid_locations) (mapf_env.py:142) */
    int32_t state_words;     /* 1 or 2 */
    int32_t moves_in_smem;   /* 1 when the per-(cell, action) move table is staged in shared memory */
    int64_t n_actions;       /* nA = 5**n (mapf_env.py:146) */
    uint64_t n_states[2];    /* nS = L**n (mapf_env.py:145), low word first */
    uint64_t start_state[2]; /* env.reset() (mapf_env.py:290-293) */
    uint64_t goal_state[2];  /* locations_to_state(agents_goals) (mapf_env.py:158) */
    int64_t max_row_len;     /* 3**n */
    int32_t device;
    int32_t sm_count;
} mapf_info;

typedef struct mapf_ctx mapf_ctx;

/* MapfEnv.__init__ (mapf_env.py:116-161): validates starts/goals, numbers the free cells, builds the obstacle
 * bitmap and -- on the device, from the bitmap staged in shared memory -- the per-(cell, action) move table that
 * `single_agent_movements` (mapf_env.py:163-184) would produce.  Synchronous. */
int mapf_ctx_create(const mapf_spec *spec, int device, mapf_ctx **out);
void mapf_ctx_destroy(mapf_ctx *ctx);
int mapf_ctx_info(const mapf_ctx *ctx, mapf_info *out);

/* single_agent_movements for every (cell, action) (mapf_env.py:163-184), read back from the device table.
 * HOST outputs: k[L*5] merged-outcome counts, dest[L*5*3] next cells (-1 padded), prob[L*5*3] (0 padded),
 * cells_rc[L*2] = valid_locations (mapf_env.py:142).  Any output may be NULL.  Synchronous. */
int mapf_ctx_moves(const mapf_ctx *ctx, uint8_t *k, int32_t *dest, double *prob, int32_t *cells_rc);

/* state_to_locations / locations_to_state in bulk (mapf_env.py:358-371, envs/__init__.py:50-79).
 * cells is int32[B*n_agents]. */
int mapf_decode_states(const mapf_ctx *ctx, const void *states, int64_t B, int32_t *cells, void *stream);
int mapf_encode_states(const mapf_ctx *ctx, const int32_t *cells, int64_t B, void *states, void *stream);

/* len(P[s][a]) for B (state, action) pairs (mapf_env.py:448-479): 1 for a terminal state, else the product of
 * the per-agent merged-outcome counts.  row_len is int64[B]. */
int mapf_count_rows(const mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B, int64_t *row_len,
                    void *stream);

/* Exclusive scan of row_len[B] into row_ptr[B+1] (row_ptr[B] = total records).  scratch: at least
 * mapf_scan_scratch_bytes(B) bytes of device memory. */
int64_t mapf_scan_scratch_bytes(int64_t B);
int mapf_scan_rows(const mapf_ctx *ctx, const int64_t *row_len, int64_t B, int64_t *row_ptr, void *scratch,
                   void *stream);

/* mapf_count_rows + mapf_scan_rows in one call (one launch and one pass over row_len fewer): row_len[B] and
 * row_ptr[B+1] are both written.  row_len may be NULL when only row_ptr is wanted: the lengths then stay in the scratch
 * as 16- or 32-bit values (8 instead of 16 bytes per row between the two passes).  The _range form does the same for a
 * table slab. */
int mapf_count_scan_rows(const mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B, int64_t *row_len,
                         int64_t *row_ptr, void *scratch, void *stream);
int mapf_count_scan_range(const mapf_ctx *ctx, const uint64_t s_begin[2], int64_t n_states, int64_t *row_len,
                          int64_t *row_ptr, void *scratch, void *stream);

/* P[s][a] for B pairs as CSR records in itertools.product order, agent 0 slowest (mapf_env.py:448-479):
 * record row_ptr[b] + j is the j-th element of P[states[b]][actions[b]].
 * next_state: state_words*8 bytes per record; prob, reward: f64; flags: MAPF_FLAG_DONE | MAPF_FLAG_COLLISION. */
int mapf_expand(const mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B, const int64_t *row_ptr,
                void *next_state, double *prob, double *reward, uint8_t *flags, void *stream);

/* The same rows for the table slab [s_begin, s_begin + n_states) x [0, nA), generated on the device without
 * per-row inputs; row index = (s - s_begin) * nA + a.  Used with mapf_count_range + mapf_scan_rows. */
int mapf_count_range(const mapf_ctx *ctx, const uint64_t s_begin[2], int64_t n_states, int64_t *row_len, void *stream);
int mapf_expand_range(const mapf_ctx *ctx, const uint64_t s_begin[2], int64_t n_states, const int64_t *row_ptr,
                      void *next_state, double *prob, double *reward, uint8_t *flags, void *stream);

/* Checksums of n_records records, accumulated (added, mod 2**64) into the device array out8[8]:
 * count, collisions, dones, sum next_state low word, sum next_state high word, sum prob bit patterns,
 * sum reward bit patterns, sum over records of (index_base + i + 1) * (next_low + 1 + 2*collision + 4*done). */
int mapf_checksum(const mapf_ctx *ctx, int64_t n_records, int64_t index_base, const void *next_state,
                  const double *prob, const double *reward, const uint8_t *flags, uint64_t *out8, void *stream);

/* MapfEnv.step for B independent envs (mapf_env.py:237-266).
 * uniforms != NULL: f64[B*n_agents], the draw `categorical_sample` would make for each agent (mapf_env.py:255) --
 *   bit-exact replay of a reference trace.
 * uniforms == NULL: Philox4x32-10 keyed by `seed`, counter (env_offset + env index, step_index, draw block); each
 *   agent uses one 32-bit word w as u = w * 2**-32.  env_offset is the index of this batch's first env in the
 *   caller's global batch, so that shards of one batch (multi-GPU, pipelined halves) draw disjoint streams.
 * A terminal state is a no-op: next_state = state, reward 0, prob 0, done 1 (mapf_env.py:238-240).
 * next_states may alias states.  done / collision are one byte each (0/1). */
int mapf_step(const mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B, const double *uniforms,
              uint64_t seed, uint64_t step_index, int64_t env_offset, uint32_t options, void *next_states,
              double *reward, double *prob, uint8_t *done, uint8_t *collision, void *stream);

/* The 64 rewards a step can return, indexed by the code MAPF_OPT_COMPACT writes: code = 16 * kind + parked agents, kind
 * 0 living, 1 clash + living, 2 goal + living, 3 step from a terminal state (0); `parked` counts the agents standing on
 * their goal that chose STAY under the sum-of-costs criterion (mapf_env.py:441-446; 0 under Makespan). */
int mapf_ctx_reward_table(const mapf_ctx *ctx, double out64[64]);

/* T consecutive steps of B envs in one launch; state lives in registers between steps.
 * actions: int32[T*B] (step-major) or NULL for a uniformly random joint action per env and step (Philox).
 * Outputs are step-major [T*B]; states_inout receives the final states.  Step t uses step_index0 + t. */
int mapf_rollout(const mapf_ctx *ctx, void *states_inout, const int32_t *actions, int64_t T, int64_t B,
                 const double *uniforms, uint64_t seed, uint64_t step_index0, int64_t env_offset, uint32_t options,
                 void *next_states, double *reward, double *prob, uint8_t *done, uint8_t *collision, void *stream);

/* ---- closed-loop policy evaluation --------------------------------------------------------------------------- */

/* outcome of an episode: the kind of its last step, or TIMEOUT when no step within max_steps was done */
enum { MAPF_EPISODE_TIMEOUT = 0, MAPF_EPISODE_COLLISION = 1, MAPF_EPISODE_GOAL = 2, MAPF_EPISODE_TERMINAL_START = 3 };
/* policy kinds of mapf_evaluate */
enum {
    MAPF_POLICY_RANDOM = 0, /* a uniformly random joint action per step, drawn as mapf_rollout draws it (policy unused) */
    MAPF_POLICY_JOINT = 1,  /* int32 policy[policy_len], indexed by the joint state (policy_len >= nS; one-word states) */
    MAPF_POLICY_AGENTS = 2, /* uint8 policy[n_agents * L]: agent i on cell c intends action policy[i * L + c] */
    MAPF_POLICY_GROUPS = 3, /* int32 tables of agent groups, one per group (mapf_evaluate_groups) */
    MAPF_POLICY_TABLE = 4   /* the actions of a value table, group tables where it has none (mapf_evaluate_table) */
};
/* conflict[e] of mapf_evaluate_groups for an episode that did not end in a collision */
#define MAPF_NO_CONFLICT 0xFF

/* Bytes of device scratch mapf_evaluate needs (its work counter).  Concurrent calls need separate scratch. */
int64_t mapf_evaluate_scratch_bytes(void);
/* n_episodes closed-loop episodes of a policy in one launch.  Episode e is exactly
 *     s = start state; G = 0; disc = 1
 *     for t in range(max_steps):
 *         a = policy(s); s, r, done = mapf_step(s, a) with Philox counter (episode_offset + e, step_index0 + t), no auto-reset
 *         G = G + disc * r; disc = disc * gamma        (single binary64 operations, no fused multiply-add)
 *         if done: break
 * i.e. env e of a mapf_step batch with env_offset = episode_offset, cut at its first done.  ret[e] = G (f64),
 * length[e] = t + 1 (int32), outcome[e] = MAPF_EPISODE_*.  Nothing is stored per step.  Out-of-range policy entries are
 * clamped.  Device sampling only: a context whose slip probabilities do not add up to 1 is MAPF_ERR_UNSUPPORTED.
 * Rejected (MAPF_ERR_INVALID): NULL pointers, max_steps < 1 or >= 2**31, n_episodes < 0 or > 2**30, AGENTS with
 * policy_len != n_agents * L, JOINT with policy_len < nS; JOINT on a two-word context is MAPF_ERR_UNSUPPORTED.
 * n_episodes == 0 launches nothing.  `scratch` (mapf_evaluate_scratch_bytes) is reset on `stream` by the call. */
int mapf_evaluate(const mapf_ctx *ctx, int32_t policy_kind, const void *policy, int64_t policy_len, int64_t n_episodes,
                  int64_t max_steps, double gamma, uint64_t seed, uint64_t step_index0, int64_t episode_offset,
                  void *scratch, double *ret, int32_t *length, uint8_t *outcome, void *stream);

/* mapf_evaluate for a product of group policies, with the pair of agents each collision episode is attributed to.
 * group_of (HOST, n_agents entries) splits the agents into groups numbered canonically: group_of[0] = 0, and each
 * further group takes the next id in the order of its lowest agent.  Group g with agents g_0 < g_1 < ... acts by
 * int32 table_g[L**|g|]: in joint state s it takes the group joint action
 *     table_g[sum_k cell(s, g_k) * L**k]        (the local state mapf_project_states(ctx, s, g) computes)
 * and agent g_k intends digit k of it, base 5 -- so table_g is the policy value iteration returns on the agent-subset
 * env of g.  `tables` (DEVICE) is table_0, table_1, ... concatenated, tables_len = sum_g L**|g| entries.  Singleton
 * groups act like MAPF_POLICY_AGENTS, one group of every agent like MAPF_POLICY_JOINT.  Episode e is exactly
 *     s = start state; G = 0; disc = 1
 *     for t in range(max_steps):
 *         a = sum_i 5**i * digit(table_{group_of[i]}[local state of group_of[i] in s], position of i in its group)
 *         s_prev = s; s, r, done = mapf_step(s, a) with Philox counter (episode_offset + e, step_index0 + t), no auto-reset
 *         G = G + disc * r; disc = disc * gamma        (single binary64 operations, no fused multiply-add)
 *         if done: break
 * with ret / length / outcome as in mapf_evaluate (same draws, queue and scratch; out-of-range entries are clamped to
 * 5**|g| - 1).  conflict (DEVICE, may be NULL): for an episode whose outcome is MAPF_EPISODE_COLLISION,
 * conflict[e] = i | j << 4 for the lexicographically smallest pair i < j that clashed in its last step (next_i == next_j,
 * or next_i == prev_j and next_j == prev_i), where pairs of agents in different groups come before pairs inside one
 * group; MAPF_NO_CONFLICT for every other episode.
 * Rejected (MAPF_ERR_INVALID): the arguments mapf_evaluate rejects, a NULL group_of or tables, a group_of that is not
 * canonical or has an id outside [0, n_agents), and tables_len != sum_g L**|g| (or a sum that overflows int64).
 * A context whose slip probabilities do not add up to 1 is MAPF_ERR_UNSUPPORTED. */
int mapf_evaluate_groups(const mapf_ctx *ctx, const int32_t *group_of, const int32_t *tables, int64_t tables_len,
                         int64_t n_episodes, int64_t max_steps, double gamma, uint64_t seed, uint64_t step_index0,
                         int64_t episode_offset, void *scratch, double *ret, int32_t *length, uint8_t *outcome,
                         uint8_t *conflict, void *stream);

/* Host-buffer convenience call (end-to-end path): copies states/actions from HOST memory, steps, copies the five
 * results back to HOST memory, on the context's own streams; returns when the results are in host memory. */
int mapf_step_host(mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B, const double *uniforms,
                   uint64_t seed, uint64_t step_index, int64_t env_offset, uint32_t options, void *next_states,
                   double *reward, double *prob, uint8_t *done, uint8_t *collision);

/* mapf_step_host for envs whose states are RESIDENT on the device, as the reference's are in the env object: MapfEnv.step
 * receives only the action and keeps self.s itself (mapf_env.py:237, 264).  states_dev is DEVICE memory of the context's GPU
 * holding the B current states; it is read and overwritten in place with the next states (under MAPF_OPT_AUTO_RESET the
 * start state for an env that was done), which are also written to the host buffer next_states, like the other four
 * results.  Only the actions cross the host link on the way in: 4 instead of 4 + 8 * words bytes per env.  All other
 * arguments, options and results are those of mapf_step_host and the results are bit-identical to it.  The call runs on the
 * context's own streams: work that produced states_dev must have completed before it is made; it returns when the results
 * are in host memory and states_dev is updated. */
int mapf_step_host_resident(mapf_ctx *ctx, void *states_dev, const int32_t *actions, int64_t B, const double *uniforms,
                            uint64_t seed, uint64_t step_index, int64_t env_offset, uint32_t options, void *next_states,
                            double *reward, double *prob, uint8_t *done, uint8_t *collision);

/* ---- rows next to the hot path (SURVEY.md 8f) ------------------------------------------------------------------ */

/* The consumer loop of a planner over the table, without materialising it:
 *     Q[b] = 0;  for ((p, collision), s2, r, done) in P[states[b]][actions[b]]:  Q[b] += p * (r + gamma * V[s2])
 * (mapf_env.py:448-479 provides P; the loop is the value-iteration backup gym-mapf's downstream planners run).
 * Every operation is one IEEE binary64 operation in exactly this order (no fused multiply-add), so the result
 * is bit-identical to the Python loop.  V is f64[v_len], indexed by the joint state: v_len >= nS is required and
 * contexts whose states need two words are rejected (MAPF_ERR_UNSUPPORTED).  Q is f64[B]. */
int mapf_backup(const mapf_ctx *ctx, const void *states, const int32_t *actions, int64_t B, const double *V,
                int64_t v_len, double gamma, double *Q, void *stream);
/* The same for the slab [s_begin, s_begin + n_states) x [0, nA): Q[(s - s_begin) * nA + a]. */
int mapf_backup_range(const mapf_ctx *ctx, const uint64_t s_begin[2], int64_t n_states, const double *V, int64_t v_len,
                      double gamma, double *Q, void *stream);
/* V_out[i] = max_a Q[i * nA + a], policy[i] = the first action attaining it (np.argmax); either output may be NULL. */
int mapf_greedy(const mapf_ctx *ctx, const double *Q, int64_t n_states, double *V_out, int32_t *policy, void *stream);

/* The exchange step of SHARDED value iteration fused into the same kernel: the new value of state s_begin + i is
 * written straight into every rank's copy of the value vector, peer_values[r][s_begin + i] (HOST array of n_peers
 * device pointers, the other ranks' being peer-mapped over NVLink, e.g. torch symmetric memory), instead of a
 * separate all-gather after the sweep.  The caller synchronises the ranks before the vector is read again. */
int mapf_greedy_bcast(const mapf_ctx *ctx, const double *Q, int64_t n_states, int64_t s_begin, double *const *peer_values,
                      int32_t n_peers, int32_t *policy, void *stream);

/* ---- real-time dynamic programming (RTDP) over a sparse value table; one-word states only ---------------------- */

/* A value table: a HOST struct of DEVICE pointers, all owned by the caller (the library never allocates or frees them).
 * Open addressing with linear probing over `capacity` slots keyed by the one-word joint state; the home slot of key s
 * is splitmix64_finalizer(s) & (capacity - 1).  Entries are never deleted.  Before its first use the caller sets every
 * key to MAPF_VTABLE_EMPTY and *count to 0.  *count holds the number of occupied slots; a store that would take more
 * than capacity / 2 slots is dropped and sets bit 63 of *count (MAPF_VTABLE_REFUSED), which stays set.  The calls below
 * are asynchronous on their stream: read *count after the stream has reached them. */
#define MAPF_VTABLE_EMPTY 0xFFFFFFFFFFFFFFFFull
#define MAPF_VTABLE_REFUSED 0x8000000000000000ull
typedef struct mapf_vtable {
    uint64_t *keys;     /* capacity slots; MAPF_VTABLE_EMPTY = free */
    double *values;     /* capacity: the value stored with the key */
    int32_t *actions;   /* capacity: the greedy joint action stored with the value */
    int64_t capacity;   /* a power of two, >= 64 */
    uint64_t *count;    /* one word: occupied slots | MAPF_VTABLE_REFUSED once a store was dropped */
} mapf_vtable;

/* The heuristic of the table calls: group_of (HOST) and hvalues (DEVICE f64[hvalues_len]) follow mapf_evaluate_groups'
 * group_of and tables -- canonical group ids, table_g of L**|g| doubles indexed by g's local state, concatenated in
 * group order, hvalues_len = sum_g L**|g| -- with values in place of actions.  For a one-word state s
 *     h(s) = 0.0 when s is terminal (two agents on one cell, or every agent on its goal), else
 *     h(s) = ((0.0 + table_0[l_0(s)]) + table_1[l_1(s)]) + ...     (group order, single binary64 additions)
 *     value_of(s) = the value stored with s when s is a key of the table, else h(s).
 * Rejected (MAPF_ERR_INVALID) by every call below: a NULL table or table pointer, a capacity that is not a power of two
 * or is below 64, B < 0, NULL or misaligned (not 8-byte) state arrays, the group_of / length errors of
 * mapf_evaluate_groups.  A context whose states take two words is MAPF_ERR_UNSUPPORTED. */

/* The Bellman update of B states over the table, with the max over actions folded in (no Q buffer exists):
 *     v_out[b] = max_a Q(states[b], a),  a_out[b] = the first action attaining it (np.argmax)
 *     Q(s, a) = 0;  for ((p, collision), s2, r, done) in P[s][a]:  Q += p * (r + gamma * value_of(s2))
 * every operation one IEEE binary64 operation in this order (mapf_backup's sum with V[s2] replaced by value_of(s2)).
 * The table is only read: the outputs do not depend on how the launch is scheduled. */
int mapf_rtdp_backup(const mapf_ctx *ctx, const void *states, int64_t B, const int32_t *group_of, const double *hvalues,
                     int64_t hvalues_len, const mapf_vtable *table, double gamma, double *v_out, int32_t *a_out,
                     void *stream);
/* Stores (states[b], v[b], a[b]) for b < B, overwriting the value and action of a key that is already present.  The
 * states of one call must be distinct.  Stores that do not fit are dropped as described at mapf_vtable. */
int mapf_vtable_store(const mapf_ctx *ctx, const void *states, int64_t B, const double *v, const int32_t *a,
                      const mapf_vtable *table, void *stream);
/* v_out[b] = value_of(states[b]); a_out[b] = the action stored with states[b], or -1 when it is not a key. */
int mapf_vtable_lookup(const mapf_ctx *ctx, const void *states, int64_t B, const int32_t *group_of, const double *hvalues,
                       int64_t hvalues_len, const mapf_vtable *table, double *v_out, int32_t *a_out, void *stream);
/* mapf_evaluate_groups with the MAPF_POLICY_TABLE policy: in state s an episode takes the action stored with s when s
 * is a key of the table, else the group action of `tables` exactly as mapf_evaluate_groups takes it.  Draws, queue,
 * scratch, ret / length / outcome and conflict are those of mapf_evaluate_groups, and so are its rejections. */
int mapf_evaluate_table(const mapf_ctx *ctx, const mapf_vtable *table, const int32_t *group_of, const int32_t *tables,
                        int64_t tables_len, int64_t n_episodes, int64_t max_steps, double gamma, uint64_t seed,
                        uint64_t step_index0, int64_t episode_offset, void *scratch, double *ret, int32_t *length,
                        uint8_t *outcome, uint8_t *conflict, void *stream);

/* MapfEnv.predecessors (mapf_env.py:373-376, 414-434) for B states as CSR: row_len[b] = |predecessors(states[b])|;
 * after mapf_scan_rows, pred[row_ptr[b] ..] holds the set (state_words * 8 bytes each, cartesian-product order with
 * agent 0 slowest; the reference returns an unordered set). */
int mapf_count_predecessors(const mapf_ctx *ctx, const void *states, int64_t B, int64_t *row_len, void *stream);
int mapf_predecessors(const mapf_ctx *ctx, const void *states, int64_t B, const int64_t *row_ptr, void *pred,
                      void *stream);

/* get_local_view (utils.py:138-157) for states: out[b] = the joint state of the sub-env made of `agents` (HOST array
 * of n_sub distinct agent indices, in the sub-env's agent order) that corresponds to states[b].  An output state has
 * mapf_projected_words(ctx, n_sub) 64-bit words (1 when L**n_sub < 2**63, else 2). */
int mapf_projected_words(const mapf_ctx *ctx, int32_t n_sub);
int mapf_project_states(const mapf_ctx *ctx, const void *states, int64_t B, const int32_t *agents, int32_t n_sub,
                        void *out_states, void *stream);

/* ---- on-disk formats and heterogeneous batches (SURVEY.md 8f row 4) ------------------------------------------- */

/* parse_map_file + MapfGrid.__init__ (utils.py:33-37, grid.py:9-25) on the DEVICE: `map_text` (HOST memory, the raw
 * bytes of a MovingAI .map file) is copied to the device, where one kernel finds the lines, drops the 4 header lines,
 * strip()s each grid row and classifies its characters.  *height / *width receive the grid size; `obstacles` (HOST,
 * may be NULL, capacity obstacles_cap bytes) the row-major cells, 1 = '@'.  A character other than '.' / '@' returns
 * MAPF_ERR_KEY with the character as the message (the reference's KeyError, grid.py:21).  Synchronous. */
int mapf_parse_map_text(const char *map_text, int64_t map_len, int device, int32_t *height, int32_t *width,
                        uint8_t *obstacles, int64_t obstacles_cap);

/* parse_scen_file (utils.py:8-30) for a file's CONTENTS, on the host (a scenario contributes at most n_agents short
 * lines): the first line is skipped; every further line must hold exactly nine tab-separated fields (the reference's
 * tuple unpacking raises ValueError otherwise -> MAPF_ERR_INVALID), fields 4..7 are int()ed and stored AS (row, col) of
 * the start and the goal; reading stops after n_agents lines or at the end of the text.  start_rc / goal_rc: HOST,
 * 2*n_agents ints each; *n_found = agents read (the reference truncates n_agents to it, utils.py:123).  No device
 * is touched. */
int mapf_parse_scen_text(const char *scen_text, int64_t scen_len, int32_t n_agents, int32_t *start_rc, int32_t *goal_rc,
                         int32_t *n_found);

/* create_mapf_env for file CONTENTS (utils.py:119-135): the map text goes through mapf_parse_map_text, the scenario
 * text through parse_scen_file's rules (utils.py:8-30: first line skipped, nine tab-separated fields per line, fields
 * 4..7 used as (row, col) of start and goal, the first n_agents lines, n_agents truncated to what the file holds),
 * then mapf_ctx_create.  Both texts are HOST memory. */
int mapf_ctx_create_from_text(const char *map_text, int64_t map_len, const char *scen_text, int64_t scen_len,
                              int32_t n_agents, double fail_prob, double reward_of_clash, double reward_of_goal,
                              double reward_of_living, int32_t criterion, int device, mapf_ctx **out);

/* What a context was built from: grid size, row-major obstacle bytes (HOST, height*width), and the (row, col) of every
 * agent's start and goal (HOST, 2*n_agents ints each).  Any output may be NULL. */
int mapf_ctx_grid(const mapf_ctx *ctx, int32_t *height, int32_t *width, uint8_t *obstacles, int32_t *start_rc,
                  int32_t *goal_rc);

/* A heterogeneous env batch: env_counts[i] envs of spec ctxs[i], concatenated in this order (spec i owns the envs
 * [sum(env_counts[:i]), sum(env_counts[:i+1]))).  All specs must live on one device and agree in agent count and
 * state width, and their move tables must be staged in shared memory (mapf_info.moves_in_smem); anything else is
 * MAPF_ERR_UNSUPPORTED -- step such specs with their own mapf_step.  The contexts must outlive the group. */
typedef struct mapf_group mapf_group;
int mapf_group_create(mapf_ctx *const *ctxs, const int64_t *env_counts, int32_t n_specs, mapf_group **out);
void mapf_group_destroy(mapf_group *group);
int64_t mapf_group_size(const mapf_group *group);
/* MapfEnv.step (mapf_env.py:237-266) for every env of the group in ONE launch; buffers and semantics as mapf_step
 * without options, indexed by the env's position in the concatenated batch (which also keys its Philox stream).
 * The one option bit it takes is MAPF_OPT_AUTO_RESET; any other bit (MAPF_OPT_COMPACT, MAPF_OPT_SHARE_SM) is
 * MAPF_ERR_UNSUPPORTED and launches nothing -- step with mapf_step for the compact layout. */
int mapf_group_step(const mapf_group *group, const void *states, const int32_t *actions, const double *uniforms,
                    uint64_t seed, uint64_t step_index, int64_t env_offset, uint32_t options, void *next_states,
                    double *reward, double *prob, uint8_t *done, uint8_t *collision, void *stream);

const char *mapf_last_error(void);
const char *mapf_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MAPF_B200_H */
