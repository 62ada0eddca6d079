// spectrum.cuh -- the k-mer abundance spectrum (count of counts) binned where the groups are known, instead of written out:
// hist[c] (1 <= c < hist_len) = number of distinct k-mers counted exactly c times; the groups with count >= hist_len go
// to a tail of (k-mer, count) pairs on the DevStatus::n_distinct cursor.  Nearly every group falls into the first few bins,
// so one global atomic per group would serialise on hist[1] (~1.5 G same-address atomics/s): a warp first merges its equal
// counts (__match_any_sync), small bins are summed per CTA in shared memory and flushed once at the end of the kernel.
#pragma once
#include "kernels.cuh"

namespace kmer {

constexpr int SPEC_SBINS = 64;   // bins 0..63 are summed in shared memory (256 bytes per CTA)

__device__ __forceinline__ void spec_reds_add32(uint32_t a, uint32_t v) {
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

// Warp-collective: every lane of the warp calls it; cnt == 0 means "no group on this lane".  s_hist: shared address of
// SPEC_SBINS uint32 bins.
__device__ __forceinline__ void spectrum_bin_warp(uint32_t s_hist, const SpecOut& o, DevStatus* status, uint64_t code, uint64_t cnt) {
    const uint32_t lane = threadIdx.x & 31u;
    const bool to_tail = cnt != 0 && cnt >= o.hist_len;
    const uint32_t tm = __ballot_sync(0xffffffffu, to_tail);
    if (tm) {
        const int leader = __ffs(tm) - 1;
        unsigned long long base = 0;
        if ((int)lane == leader) base = atomicAdd(&status->n_distinct, (unsigned long long)__popc(tm));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (to_tail) {
            const unsigned long long idx = base + __popc(tm & ((1u << lane) - 1u));
            if (idx < o.tail_cap) { o.tail[idx].code = code; o.tail[idx].count = cnt; }
            else status->out_overflow = 1;
        }
    }
    const uint64_t bin = to_tail ? 0 : cnt;
    const uint32_t same = __match_any_sync(0xffffffffu, bin);
    if (bin && (int)lane == __ffs(same) - 1) {
        if (bin < (uint64_t)SPEC_SBINS) spec_reds_add32(s_hist + 4u * (uint32_t)bin, (uint32_t)__popc(same));
        else atomicAdd(&o.hist[bin], (unsigned long long)__popc(same));
    }
}

// after a barrier: the CTA's shared bins -> hist
__device__ __forceinline__ void spectrum_flush(uint32_t s_hist, const SpecOut& o) {
    for (uint32_t i = threadIdx.x; i < (uint32_t)SPEC_SBINS && i < o.hist_len; i += blockDim.x) {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(s_hist + 4u * i) : "memory");
        if (v) atomicAdd(&o.hist[i], (unsigned long long)v);
    }
}

}  // namespace kmer
