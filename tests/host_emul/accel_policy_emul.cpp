// Host build of the accelerator policy (genedex_b200/csrc/accel_policy.h) for tests/test_accel_policy_host.py.
// flags: 1 = no dense suffix array, 2 = no seed table, 4 = no row context table.  free = ~0: unknown.
#include <cstdint>

#include "../../genedex_b200/csrc/accel_policy.h"

namespace {
gdx::AccelPolicy policy(uint64_t n, uint64_t budget, uint32_t ns, uint32_t lookup_depth, int wide, int text,
                        uint32_t flags) {
    return gdx::AccelPolicy{n, budget, ns, lookup_depth, wide != 0, text != 0, (flags & 1) != 0, (flags & 2) != 0,
                            (flags & 4) != 0};
}
}  // namespace

// {dense_sa, seed_depth, row_context, row_context_possible} into out
extern "C" void emul_accel_policy(uint64_t n, uint64_t budget, uint32_t ns, uint32_t lookup_depth, int wide, int text,
                                  uint32_t flags, uint64_t used, uint64_t free, const char *env_dense,
                                  const char *env_seed, const char *env_row, uint64_t *out) {
    const gdx::AccelPolicy p = policy(n, budget, ns, lookup_depth, wide, text, flags);
    out[0] = p.dense_sa(used, free, env_dense);
    out[1] = p.seed_depth(used, free, env_seed);
    out[2] = p.row_context(used, free, env_row);
    out[3] = p.row_context_possible();
}

extern "C" uint64_t emul_seed_entries(uint32_t ns, uint32_t d) { return gdx::seed_entries(ns, d); }

extern "C" uint32_t emul_verify_min_remaining(int dense_sa, const char *env) {
    return gdx::verify_min_remaining(dense_sa != 0, env);
}
