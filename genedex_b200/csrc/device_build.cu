// device_build.cu -- see device_build.h
#include "device_build.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

namespace gdx {

namespace {

struct MaxU32 {
    __host__ __device__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};

// head marker of sorted position i: i if it starts a new key group, else 0 (max-scan propagates it)
struct HeadOfKeys {
    const uint64_t *key;
    __host__ __device__ uint32_t operator()(uint32_t i) const {
        return (i == 0 || key[i] != key[i - 1]) ? i : 0u;
    }
};
struct HeadOfRoundKeys {
    const uint64_t *key;
    const uint32_t *slots;
    __host__ __device__ uint32_t operator()(uint32_t j) const {
        return (j == 0 || key[j] != key[j - 1]) ? slots[j] : 0u;
    }
};

// key(i) = first k symbols of suffix i, `bits` bits each, code = symbol + 1, 0 beyond the end
__global__ void k_make_keys(const uint8_t *__restrict__ text, uint64_t n, uint32_t bits, uint32_t k,
                            uint64_t *__restrict__ keys, uint32_t *__restrict__ vals) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t key = 0;
    for (uint32_t j = 0; j < k; ++j) {
        const uint64_t p = i + j;
        const uint64_t code = p < n ? (uint64_t)text[p] + 1 : 0;
        key = (key << bits) | code;
    }
    keys[i] = key;
    vals[i] = (uint32_t)i;
}

// unsorted[i] = 1 unless position i is a group of its own (head[i] == i and the next one is a head)
__global__ void k_unsorted_flags(const uint32_t *__restrict__ head, uint64_t n, uint8_t *__restrict__ unsorted) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const bool is_head = head[i] == (uint32_t)i;
    const bool next_is_head = i + 1 >= n || head[i + 1] == (uint32_t)(i + 1);
    unsorted[i] = !(is_head && next_is_head);
}

__global__ void k_scatter_isa(const uint32_t *__restrict__ sa, const uint32_t *__restrict__ head, uint64_t n,
                              uint32_t *__restrict__ isa) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) isa[sa[i]] = head[i];
}

// key of an open suffix in round h: (its current group head, rank of the suffix h further on)
__global__ void k_round_keys(const uint32_t *__restrict__ slots, uint64_t m, const uint32_t *__restrict__ sa,
                             const uint32_t *__restrict__ head, const uint32_t *__restrict__ isa, uint64_t n,
                             uint64_t h, uint64_t *__restrict__ keys, uint32_t *__restrict__ vals) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint32_t i = slots[j];
    const uint32_t p = sa[i];
    const uint64_t q = (uint64_t)p + h;
    const uint64_t second = q < n ? (uint64_t)isa[q] + 1 : 0;  // shorter suffix sorts first
    keys[j] = ((uint64_t)head[i] << 32) | second;
    vals[j] = p;
}

__global__ void k_round_update(const uint32_t *__restrict__ slots, uint64_t m, const uint64_t *__restrict__ keys,
                               const uint32_t *__restrict__ vals, const uint32_t *__restrict__ newhead,
                               uint32_t *__restrict__ sa, uint32_t *__restrict__ head, uint32_t *__restrict__ isa,
                               uint8_t *__restrict__ still_open) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint32_t i = slots[j], p = vals[j], nh = newhead[j];
    sa[i] = p;
    head[i] = nh;
    isa[p] = nh;
    const bool is_head = j == 0 || keys[j] != keys[j - 1];
    const bool next_is_head = j + 1 >= m || keys[j + 1] != keys[j];
    still_open[j] = !(is_head && next_is_head);
}

// bwt.rs:93-116 + sampled_suffix_array.rs:27-54
__global__ void k_bwt_and_samples(const uint8_t *__restrict__ text, const uint32_t *__restrict__ sa, uint64_t n,
                                  uint32_t sampling_rate, uint8_t *__restrict__ bwt,
                                  uint32_t *__restrict__ samples, uint64_t *__restrict__ border_rows,
                                  uint64_t *__restrict__ border_pos, unsigned long long *border_count,
                                  uint64_t border_cap) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t p = sa[i];
    const uint8_t b = text[(p ? (uint64_t)p : n) - 1];
    bwt[i] = b;
    if (i % sampling_rate == 0) samples[i / sampling_rate] = p;
    if (b == 0) {
        const unsigned long long k = atomicAdd(border_count, 1ull);
        if (k < border_cap) {
            border_rows[k] = i;
            border_pos[k] = p;
        }
    }
}

// inverse suffix array at every s-th text position: out[SA[i] / s] = i for SA[i] % s == 0
__global__ void k_sample_isa(const uint32_t *__restrict__ sa, uint64_t n, uint32_t sampling_rate,
                             uint32_t *__restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t p = sa[i];
    if (p % sampling_rate == 0) out[p / sampling_rate] = (uint32_t)i;
}

__global__ void k_count_zeros(const uint8_t *__restrict__ text, uint64_t n, unsigned long long *out) {
    uint64_t local = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        local += text[i] == 0;
    if (local) atomicAdd(out, (unsigned long long)local);
}

// O(n) suffix array check: inv must be the inverse permutation; then suffix sa[i-1] < suffix sa[i]
// iff (T[a], rank(a+1)) < (T[b], rank(b+1)) with rank(n) = -1.
__global__ void k_verify_inverse(const uint32_t *__restrict__ sa, uint64_t n, uint32_t *__restrict__ inv) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && sa[i] < n) inv[sa[i]] = (uint32_t)i;
}
__global__ void k_verify_order(const uint8_t *__restrict__ text, const uint32_t *__restrict__ sa,
                               const uint32_t *__restrict__ inv, uint64_t n, unsigned long long *violations) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool bad = inv[i] == 0xffffffffu || sa[i] >= n;  // not a permutation
    if (!bad && i > 0) {
        const uint64_t a = sa[i - 1], b = sa[i];
        if (a >= n) {
            bad = true;
        } else {
            const uint8_t ta = text[a], tb = text[b];
            if (ta != tb) {
                bad = ta > tb;
            } else {
                const int64_t ra = a + 1 < n ? (int64_t)inv[a + 1] : -1;
                const int64_t rb = b + 1 < n ? (int64_t)inv[b + 1] : -1;
                bad = ra >= rb;
            }
        }
    }
    if (bad) atomicAdd(violations, 1ull);
}

unsigned grid_for(uint64_t n, unsigned block = 256) { return (unsigned)((n + block - 1) / block); }

}  // namespace

#define DB_TRY(expr)                                                                              \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            char _buf[512];                                                                       \
            snprintf(_buf, sizeof _buf, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),  \
                     __FILE__, __LINE__);                                                         \
            err = _buf;                                                                           \
            out = DeviceBuildResult();                                                            \
            return _e == cudaErrorMemoryAllocation ? GDX_ERR_OOM : GDX_ERR_CUDA;                  \
        }                                                                                         \
    } while (0)

gdx_status device_build_from_text(const uint8_t *h_text, const uint8_t *d_text_in, uint64_t n, uint32_t sigma,
                                  uint32_t sampling_rate, DeviceBuildResult &out, std::string &err, bool keep_sa,
                                  bool verify, bool want_isa) {
    if (n >= 0xffffffffull) {
        err = "device construction supports text lengths below 2^32 - 1";
        return GDX_ERR_UNSUPPORTED;
    }
    if (n == 0 || sampling_rate == 0) {
        err = "empty text or sampling rate 0";
        return GDX_ERR_BAD_ARG;
    }
    DevMem text_own;
    const uint8_t *text = d_text_in;
    if (!text) {
        DB_TRY(text_own.alloc(n));
        DB_TRY(cudaMemcpy(text_own.p, h_text, n, cudaMemcpyHostToDevice));
        text = text_own.as<uint8_t>();
    }
    uint32_t bits = 1;
    while ((1u << bits) < sigma + 1) ++bits;
    const uint32_t k = 64 / bits;

    // ---- phase 1: sort all suffixes by their first k symbols ---------------------------------------
    DevMem keyA, keyB, valA, valB, tmp;
    DB_TRY(keyA.alloc(n * 8));
    DB_TRY(keyB.alloc(n * 8));
    DB_TRY(valA.alloc(n * 4));
    DB_TRY(valB.alloc(n * 4));
    k_make_keys<<<grid_for(n), 256>>>(text, n, bits, k, keyA.as<uint64_t>(), valA.as<uint32_t>());
    DB_TRY(cudaGetLastError());
    cub::DoubleBuffer<uint64_t> dk(keyA.as<uint64_t>(), keyB.as<uint64_t>());
    cub::DoubleBuffer<uint32_t> dv(valA.as<uint32_t>(), valB.as<uint32_t>());
    size_t tmp_bytes = 0;
    DB_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dk, dv, (int64_t)n, 0, (int)(k * bits)));
    DB_TRY(tmp.alloc(tmp_bytes));
    DB_TRY(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, dk, dv, (int64_t)n, 0, (int)(k * bits)));

    // ---- phase 2: group heads (= ranks) from the sorted keys --------------------------------------
    DevMem head, open_flags;
    DB_TRY(head.alloc(n * 4));
    DB_TRY(open_flags.alloc(n));
    {
        using Count = cub::CountingInputIterator<uint32_t, int64_t>;
        cub::TransformInputIterator<uint32_t, HeadOfKeys, Count, int64_t> it(Count(0), HeadOfKeys{dk.Current()});
        size_t b2 = 0;
        DB_TRY(cub::DeviceScan::InclusiveScan(nullptr, b2, it, head.as<uint32_t>(), MaxU32(), (int64_t)n));
        if (b2 > tmp_bytes) {
            DB_TRY(tmp.alloc(b2));
            tmp_bytes = b2;
        }
        DB_TRY(cub::DeviceScan::InclusiveScan(tmp.p, b2, it, head.as<uint32_t>(), MaxU32(), (int64_t)n));
    }
    k_unsorted_flags<<<grid_for(n), 256>>>(head.as<uint32_t>(), n, open_flags.as<uint8_t>());
    DB_TRY(cudaGetLastError());
    DB_TRY(cudaDeviceSynchronize());
    // keep the sorted positions as SA, drop the wide key buffers before ISA is allocated
    DevMem sa;
    if (dv.Current() == valA.as<uint32_t>()) {
        sa = std::move(valA);
        valB.reset();
    } else {
        sa = std::move(valB);
        valA.reset();
    }
    keyA.reset();
    keyB.reset();
    DevMem isa;
    DB_TRY(isa.alloc(n * 4));
    k_scatter_isa<<<grid_for(n), 256>>>(sa.as<uint32_t>(), head.as<uint32_t>(), n, isa.as<uint32_t>());
    DB_TRY(cudaGetLastError());

    // ---- phase 3: doubling rounds over the still open suffixes -----------------------------------
    DevMem slots, slots2, d_m;
    DB_TRY(d_m.alloc(8));
    uint64_t m = 0;
    {
        // number of open positions first, so that the worklists can be sized
        DB_TRY(slots.alloc(n * 4));
        using Count = cub::CountingInputIterator<uint32_t, int64_t>;
        size_t b3 = 0;
        DB_TRY(cub::DeviceSelect::Flagged(nullptr, b3, Count(0), open_flags.as<uint8_t>(), slots.as<uint32_t>(),
                                          d_m.as<uint64_t>(), (int64_t)n));
        if (b3 > tmp_bytes) {
            DB_TRY(tmp.alloc(b3));
            tmp_bytes = b3;
        }
        DB_TRY(cub::DeviceSelect::Flagged(tmp.p, b3, Count(0), open_flags.as<uint8_t>(), slots.as<uint32_t>(),
                                          d_m.as<uint64_t>(), (int64_t)n));
        DB_TRY(cudaMemcpy(&m, d_m.p, 8, cudaMemcpyDeviceToHost));
    }
    open_flags.reset();
    out.rounds = 0;
    if (m > 0) {
        DevMem rkA, rkB, rvA, rvB, newhead, still_open;
        DB_TRY(rkA.alloc(m * 8));
        DB_TRY(rkB.alloc(m * 8));
        DB_TRY(rvA.alloc(m * 4));
        DB_TRY(rvB.alloc(m * 4));
        DB_TRY(newhead.alloc(m * 4));
        DB_TRY(still_open.alloc(m));
        DB_TRY(slots2.alloc(m * 4));
        for (uint64_t h = k; m > 0; h *= 2) {
            ++out.rounds;
            k_round_keys<<<grid_for(m), 256>>>(slots.as<uint32_t>(), m, sa.as<uint32_t>(), head.as<uint32_t>(),
                                               isa.as<uint32_t>(), n, h, rkA.as<uint64_t>(), rvA.as<uint32_t>());
            DB_TRY(cudaGetLastError());
            cub::DoubleBuffer<uint64_t> rk(rkA.as<uint64_t>(), rkB.as<uint64_t>());
            cub::DoubleBuffer<uint32_t> rv(rvA.as<uint32_t>(), rvB.as<uint32_t>());
            size_t b4 = 0;
            DB_TRY(cub::DeviceRadixSort::SortPairs(nullptr, b4, rk, rv, (int64_t)m, 0, 64));
            if (b4 > tmp_bytes) {
                DB_TRY(tmp.alloc(b4));
                tmp_bytes = b4;
            }
            DB_TRY(cub::DeviceRadixSort::SortPairs(tmp.p, b4, rk, rv, (int64_t)m, 0, 64));
            {
                using Count = cub::CountingInputIterator<uint32_t, int64_t>;
                cub::TransformInputIterator<uint32_t, HeadOfRoundKeys, Count, int64_t> it(
                    Count(0), HeadOfRoundKeys{rk.Current(), slots.as<uint32_t>()});
                size_t b5 = 0;
                DB_TRY(cub::DeviceScan::InclusiveScan(nullptr, b5, it, newhead.as<uint32_t>(), MaxU32(), (int64_t)m));
                if (b5 > tmp_bytes) {
                    DB_TRY(tmp.alloc(b5));
                    tmp_bytes = b5;
                }
                DB_TRY(cub::DeviceScan::InclusiveScan(tmp.p, b5, it, newhead.as<uint32_t>(), MaxU32(), (int64_t)m));
            }
            k_round_update<<<grid_for(m), 256>>>(slots.as<uint32_t>(), m, rk.Current(), rv.Current(),
                                                 newhead.as<uint32_t>(), sa.as<uint32_t>(), head.as<uint32_t>(),
                                                 isa.as<uint32_t>(), still_open.as<uint8_t>());
            DB_TRY(cudaGetLastError());
            size_t b6 = 0;
            DB_TRY(cub::DeviceSelect::Flagged(nullptr, b6, slots.as<uint32_t>(), still_open.as<uint8_t>(),
                                              slots2.as<uint32_t>(), d_m.as<uint64_t>(), (int64_t)m));
            if (b6 > tmp_bytes) {
                DB_TRY(tmp.alloc(b6));
                tmp_bytes = b6;
            }
            DB_TRY(cub::DeviceSelect::Flagged(tmp.p, b6, slots.as<uint32_t>(), still_open.as<uint8_t>(),
                                              slots2.as<uint32_t>(), d_m.as<uint64_t>(), (int64_t)m));
            DB_TRY(cudaMemcpy(&m, d_m.p, 8, cudaMemcpyDeviceToHost));
            std::swap(slots, slots2);
            if (h > (1ull << 40)) {
                err = "prefix doubling did not converge";
                out = DeviceBuildResult();
                return GDX_ERR_CUDA;
            }
        }
    }
    slots.reset();
    slots2.reset();
    head.reset();
    isa.reset();

    // ---- optional O(n) verification ------------------------------------------------------------------
    if (verify) {
        DevMem inv, viol;
        DB_TRY(inv.alloc(n * 4));
        DB_TRY(viol.alloc(8));
        DB_TRY(cudaMemset(inv.p, 0xff, n * 4));
        DB_TRY(cudaMemset(viol.p, 0, 8));
        k_verify_inverse<<<grid_for(n), 256>>>(sa.as<uint32_t>(), n, inv.as<uint32_t>());
        k_verify_order<<<grid_for(n), 256>>>(text, sa.as<uint32_t>(), inv.as<uint32_t>(), n,
                                             viol.as<unsigned long long>());
        DB_TRY(cudaGetLastError());
        DB_TRY(cudaMemcpy(&out.verify_violations, viol.p, 8, cudaMemcpyDeviceToHost));
    }

    // ---- phase 4: BWT, samples, text borders --------------------------------------------------------
    DevMem zeros;
    DB_TRY(zeros.alloc(16));
    DB_TRY(cudaMemset(zeros.p, 0, 16));
    k_count_zeros<<<148 * 8, 256>>>(text, n, zeros.as<unsigned long long>());
    DB_TRY(cudaGetLastError());
    uint64_t nzero = 0;
    DB_TRY(cudaMemcpy(&nzero, zeros.p, 8, cudaMemcpyDeviceToHost));
    const uint64_t nsamp = (n + sampling_rate - 1) / sampling_rate;
    DevMem bwt, samples, brow, bpos;
    DB_TRY(bwt.alloc(n));
    DB_TRY(samples.alloc(nsamp * 4));
    DB_TRY(brow.alloc((nzero + 1) * 8));
    DB_TRY(bpos.alloc((nzero + 1) * 8));
    k_bwt_and_samples<<<grid_for(n), 256>>>(text, sa.as<uint32_t>(), n, sampling_rate, bwt.as<uint8_t>(),
                                            samples.as<uint32_t>(), brow.as<uint64_t>(), bpos.as<uint64_t>(),
                                            zeros.as<unsigned long long>() + 1, nzero);
    DB_TRY(cudaGetLastError());
    uint64_t nborder = 0;
    DB_TRY(cudaMemcpy(&nborder, zeros.as<uint64_t>() + 1, 8, cudaMemcpyDeviceToHost));
    if (nborder != nzero) {
        err = "internal error: number of BWT sentinels differs from the number of text sentinels";
        out = DeviceBuildResult();
        return GDX_ERR_CUDA;
    }
    std::vector<uint64_t> rows(nborder), pos(nborder);
    DB_TRY(cudaMemcpy(rows.data(), brow.p, nborder * 8, cudaMemcpyDeviceToHost));
    DB_TRY(cudaMemcpy(pos.data(), bpos.p, nborder * 8, cudaMemcpyDeviceToHost));
    std::vector<uint64_t> order(nborder);
    for (uint64_t i = 0; i < nborder; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return rows[a] < rows[b]; });
    out.border_rows.resize(nborder);
    out.border_pos.resize(nborder);
    for (uint64_t i = 0; i < nborder; ++i) {
        out.border_rows[i] = rows[order[i]];
        out.border_pos[i] = pos[order[i]];
    }
    if (want_isa) {
        DevMem isa_s;
        DB_TRY(isa_s.alloc(nsamp * 4));
        k_sample_isa<<<grid_for(n), 256>>>(sa.as<uint32_t>(), n, sampling_rate, isa_s.as<uint32_t>());
        DB_TRY(cudaGetLastError());
        out.d_isa_samples = std::move(isa_s);
    }
    out.d_bwt = std::move(bwt);
    out.d_samples = std::move(samples);
    if (keep_sa) out.d_sa = std::move(sa);
    return GDX_OK;
}

}  // namespace gdx
