// device_build.h -- suffix array / BWT construction on the GPU (construction is not on the search
// path; this exists so that a 3.1 Gbp index can be built in seconds on the box that serves it).
//
// Prefix doubling with radix sorts (Manber-Myers ranks, Larsson-Sadakane style discarding of
// already sorted suffixes).  Same ordering convention as libsais as called by the reference
// (construction/mod.rs:88-103): end of text < every symbol, sentinels are ordinary symbols.  The
// suffix array of a text is unique, so this yields the reference's BWT / samples / border map;
// k_verify_suffix_array re-checks the result in O(n) when asked to.
#ifndef GDX_DEVICE_BUILD_H
#define GDX_DEVICE_BUILD_H

#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/genedex_b200.h"
#include "cuda_owners.h"

namespace gdx {

struct DeviceBuildResult {
    DevMem d_bwt;          // n bytes, dense symbols
    DevMem d_samples;      // u32 SA[0], SA[s], ... (n < 2^32 - 1)
    DevMem d_sa;           // u32 full suffix array, only when keep_sa
    DevMem d_isa_samples;  // u32 ISA[0], ISA[s], ... (row of every s-th text position), when want_isa
    std::vector<uint64_t> border_rows, border_pos;  // sorted by row (bwt.rs:108-116)
    uint64_t verify_violations = 0;                 // only meaningful when verify was requested
    uint32_t rounds = 0;
};

// exactly one of h_text / d_text is non-null (dense symbols incl. sentinels)
gdx_status device_build_from_text(const uint8_t *h_text, const uint8_t *d_text, uint64_t n, uint32_t sigma,
                                  uint32_t sampling_rate, DeviceBuildResult &out, std::string &err,
                                  bool keep_sa = false, bool verify = false, bool want_isa = false);

}  // namespace gdx
#endif
