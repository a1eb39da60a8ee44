// mapf_inst.cu -- instantiates every hot kernel for ONE agent count (compile with -DMAPF_N=<n>); the Makefile
// builds the 13 units in parallel.
#include "mapf_host.h"
#include "mapf_kernels.cuh"

#ifndef MAPF_N
#error "compile with -DMAPF_N=<agents>"
#endif

template <int N, int W, bool LUTS>
static void fill(KernelSet *k) {
    k->step_philox1 = (const void *)k_step<N, W, LUTS, false, 1>;
    k->step_tape = (const void *)k_step<N, W, LUTS, true, 1>;
    k->step_philox1c = (const void *)k_step<N, W, LUTS, false, 1, true>;
    k->step_tape_c = (const void *)k_step<N, W, LUTS, true, 1, true>;
    k->step_philox1k = (const void *)k_step<N, W, LUTS, false, 1, false, true>;
    k->step_tape_k = (const void *)k_step<N, W, LUTS, true, 1, false, true>;
    k->step_philox1ck = (const void *)k_step<N, W, LUTS, false, 1, true, true>;
    k->step_tape_ck = (const void *)k_step<N, W, LUTS, true, 1, true, true>;
    // EPT = 2; with a staged move table, from STEP_WIDE_MIN_AGENTS agents on the step runs one env per thread instead
    if constexpr (!(LUTS && N >= STEP_WIDE_MIN_AGENTS)) {
        k->step_philox2 = (const void *)k_step<N, W, LUTS, false, 2>;
        k->step_philox2c = (const void *)k_step<N, W, LUTS, false, 2, true>;
        k->step_philox2k = (const void *)k_step<N, W, LUTS, false, 2, false, true>;
        k->step_philox2ck = (const void *)k_step<N, W, LUTS, false, 2, true, true>;
    }
    k->rollout_philox = (const void *)k_rollout<N, W, LUTS, false, 1, true>;
    k->rollout_philox_rnd = (const void *)k_rollout<N, W, LUTS, false, 1, false>;
    if constexpr (N <= 6) {
        k->rollout_philox2 = (const void *)k_rollout<N, W, LUTS, false, 2, true>;
        k->rollout_philox2_rnd = (const void *)k_rollout<N, W, LUTS, false, 2, false>;
    }
    k->rollout_tape = (const void *)k_rollout<N, W, LUTS, true, 1, true>;
    k->rollout_tape_rnd = (const void *)k_rollout<N, W, LUTS, true, 1, false>;
    if (LUTS) {
        k->step_group_philox = (const void *)k_step_group<N, W, false>;
        k->step_group_tape = (const void *)k_step_group<N, W, true>;
    }
    k->expand = (const void *)k_expand<N, W, LUTS, false>;
    k->expand_range = (const void *)k_expand<N, W, LUTS, true>;
    k->count = (const void *)k_count<N, W, false, LUTS>;
    k->count_range = (const void *)k_count<N, W, true, LUTS>;
    k->count_partials = (const void *)k_count_partials<N, W, false, LUTS>;
    k->count_partials_range = (const void *)k_count_partials<N, W, true, LUTS>;
    // compact row lengths (kept in the scan's scratch when the caller does not ask for row_len): 3**10 < 2**16
    if constexpr (N <= 10) {
        k->count_partials_c = (const void *)k_count_partials<N, W, false, LUTS, u16>;
        k->count_partials_range_c = (const void *)k_count_partials<N, W, true, LUTS, u16>;
        k->compact_len_bytes = 2;
    } else {
        k->count_partials_c = (const void *)k_count_partials<N, W, false, LUTS, u32>;
        k->count_partials_range_c = (const void *)k_count_partials<N, W, true, LUTS, u32>;
        k->compact_len_bytes = 4;
    }
    k->decode = (const void *)k_decode<N, W>;
    k->encode = (const void *)k_encode<N, W>;
    if (W == 1) {
        k->backup = (const void *)k_backup<N, LUTS, false>;
        k->backup_range = (const void *)k_backup<N, LUTS, true>;
        k->rtdp_backup = (const void *)k_rtdp_backup<N, LUTS>;
        k->vtable_lookup = (const void *)k_vtable_lookup<N>;
        k->evaluate_table = (const void *)k_evaluate_table<N, LUTS>;
    }
    k->evaluate[0] = (const void *)k_evaluate<N, W, LUTS, 0>;
    if constexpr (W == 1) k->evaluate[1] = (const void *)k_evaluate<N, W, LUTS, 1>;  // policy indexed by the joint state
    k->evaluate[2] = (const void *)k_evaluate<N, W, LUTS, 2>;
    k->evaluate[3] = (const void *)k_evaluate_groups<N, W, LUTS>;
    k->pred_count = (const void *)k_pred_count<N, W>;
    k->pred_emit = (const void *)k_pred_emit<N, W>;
    k->project = (const void *)k_project<N, W>;
    k->expand_slab_bytes = sizeof(ExpandSlab<N>);
    k->expand_threads = LUTS ? EXPAND_THREADS(N) : 0;  // 0: the context's CTA size
    k->step_threads = LUTS && N >= STEP_WIDE_MIN_AGENTS ? STEP_WIDE_THREADS : 0;  // != 0: one env per thread, wide CTAs
    k->backup_slab_bytes = sizeof(BackupSlab<N>);
}

#define CAT_(a, b) a##b
#define CAT(a, b) CAT_(a, b)

void CAT(mapf_get_kernels_, MAPF_N)(int words, int luts, KernelSet *out) {
    // two-word states need L**n >= 2**63 with L <= 65535, i.e. at least 4 agents
    if (words == 1) {
        if (luts) fill<MAPF_N, 1, true>(out);
        else fill<MAPF_N, 1, false>(out);
    } else {
#if MAPF_N >= 4
        if (luts) fill<MAPF_N, 2, true>(out);
        else fill<MAPF_N, 2, false>(out);
#else
        (void)out;
#endif
    }
}
