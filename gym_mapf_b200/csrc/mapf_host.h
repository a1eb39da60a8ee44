// mapf_host.h -- glue between the per-agent-count kernel instantiation units (mapf_inst.cu, compiled once per N)
// and the C ABI (mapf_capi.cu).
#pragma once
#include <cstddef>

struct KernelSet {
    const void *step_philox1 = nullptr;  // k_step<N, W, LUTS, TAPE=false, EPT=1>
    const void *step_philox2 = nullptr;  // ... EPT=2 (128-bit I/O); null when step_threads != 0
    const void *step_tape = nullptr;     // k_step<N, W, LUTS, TAPE=true, EPT=1>
    const void *step_philox1c = nullptr, *step_philox2c = nullptr, *step_tape_c = nullptr;  // ... COMPACT outputs
    // ... KEEP = true (mapf_step_host_resident: next states also stored to the device-resident array), plain / COMPACT
    const void *step_philox1k = nullptr, *step_philox2k = nullptr, *step_tape_k = nullptr;
    const void *step_philox1ck = nullptr, *step_philox2ck = nullptr, *step_tape_ck = nullptr;
    const void *rollout_philox = nullptr, *rollout_tape = nullptr;  // k_rollout<N, W, LUTS, TAPE, EPT=1>
    const void *rollout_philox2 = nullptr;                            // ... EPT=2 (128-bit stores)
    const void *rollout_philox_rnd = nullptr, *rollout_philox2_rnd = nullptr, *rollout_tape_rnd = nullptr;  // actions == NULL
    const void *step_group_philox = nullptr, *step_group_tape = nullptr;  // k_step_group<N, W, TAPE>; staged move tables only
    const void *expand = nullptr, *expand_range = nullptr;
    const void *count = nullptr, *count_range = nullptr;
    const void *count_partials = nullptr, *count_partials_range = nullptr;  // row lengths + the scan's chunk sums
    const void *count_partials_c = nullptr, *count_partials_range_c = nullptr;  // ... with u16 / u32 lengths
    int compact_len_bytes = 0;
    const void *decode = nullptr, *encode = nullptr;
    const void *backup = nullptr, *backup_range = nullptr;  // k_backup<N, LUTS, RANGE>; one-word states only
    // by MAPF_POLICY_* kind: k_evaluate<N, W, LUTS, POLICY> for 0..2, k_evaluate_groups<N, W, LUTS> for 3
    const void *evaluate[4] = {nullptr, nullptr, nullptr, nullptr};
    // RTDP over a value table (one-word states only): k_rtdp_backup<N, LUTS>, k_vtable_lookup<N>, k_evaluate_table<N, LUTS>
    const void *rtdp_backup = nullptr, *vtable_lookup = nullptr, *evaluate_table = nullptr;
    const void *pred_count = nullptr, *pred_emit = nullptr, *project = nullptr;
    size_t expand_slab_bytes = 0;        // per warp
    int expand_threads = 0;              // CTA size of k_expand (0: the context's)
    int step_threads = 0;                // CTA size of the EPT = 1 k_step kernels, which are then always used (0: the context's)
    size_t backup_slab_bytes = 0;        // per warp
};

// words: 1 or 2; luts: move table staged in shared memory
typedef void (*mapf_kernels_fn)(int words, int luts, KernelSet *out);
#define DECL(N) void mapf_get_kernels_##N(int words, int luts, KernelSet *out);
DECL(1) DECL(2) DECL(3) DECL(4) DECL(5) DECL(6) DECL(7) DECL(8) DECL(9) DECL(10) DECL(11) DECL(12) DECL(13)
#undef DECL
