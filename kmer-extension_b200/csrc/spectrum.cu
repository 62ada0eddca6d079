// spectrum.cu -- the abundance spectrum of a table that already exists in HBM: the tier-2 / global hash table (hash_compact's
// input), the dense 4^k counters (dense_compact's input) or a (k-mer, count) pair array.  One pass over the table; nothing
// is written per group except the tail (spectrum.cuh).
#include "spectrum.cuh"

namespace kmer {

enum SpecSrc { SPEC_PAIRS = 0, SPEC_HASH = 1, SPEC_DENSE = 2 };

// SPEC_HASH: slots hold (code, count - 1), empty = kEmpty; gated: tier 2's table, only read if the device ran tier 2
// (DevStatus::t2_mode == 1); the k == 32 special key (DevStatus::special_count) is binned either way, as hash_compact appends it.
// SPEC_DENSE: in[b] = count of code b; only the bins b % n_ranks == rank.
// SPEC_PAIRS: (code, count) pairs.
template <int SRC>
__global__ void __launch_bounds__(256) spectrum_scan_kernel(const void* __restrict__ in, uint64_t n, int k, SpecOut o, DevStatus* status,
                                                            int gated, uint32_t rank, uint32_t n_ranks) {
    __shared__ uint32_t s_hist[SPEC_SBINS];
    for (int i = threadIdx.x; i < SPEC_SBINS; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    const uint32_t hs = smem_u32(s_hist);
    const int lane = threadIdx.x & 31;
    if (SRC == SPEC_HASH && gated) n = status->t2_mode == 1ull ? status->t2_slots : 0;
    const uint64_t n32 = (n + 31) & ~31ull;                           // whole warps: spectrum_bin_warp is warp-collective
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    unsigned long long total = 0;
    for (uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; b < n32; b += stride) {
        uint64_t code = 0, cnt = 0;
        if (b < n) {
            if (SRC == SPEC_DENSE) {
                if (n_ranks <= 1 || b % n_ranks == rank) { code = b; cnt = reinterpret_cast<const unsigned long long*>(in)[b]; }
            } else {
                const uint4 raw = ld_nc_u128(reinterpret_cast<const kmer_count_pair*>(in) + b);
                code = ((uint64_t)raw.y << 32) | raw.x;
                cnt = ((uint64_t)raw.w << 32) | raw.z;
                if (SRC == SPEC_HASH) cnt = code != kEmpty ? cnt + 1 : 0;
            }
        }
        total += cnt;
        spectrum_bin_warp(hs, o, status, code, cnt);
    }
    for (int d = 16; d; d >>= 1) total += __shfl_xor_sync(0xffffffffu, total, d);
    if (lane == 0 && total) atomicAdd(&status->n_kmers, total);
    if (SRC == SPEC_HASH && k == 32 && blockIdx.x == 0 && threadIdx.x < 32) {   // the one key that cannot live in the table
        const unsigned long long sc = status->special_count;
        spectrum_bin_warp(hs, o, status, kEmpty, threadIdx.x == 0 ? sc : 0ull);
        if (threadIdx.x == 0 && sc) atomicAdd(&status->n_kmers, sc);
    }
    __syncthreads();
    spectrum_flush(hs, o);
}

static unsigned scan_blocks(const DeviceInfo& di, uint64_t n) {
    uint64_t blocks = (n + 255) / 256;
    const uint64_t maxb = (uint64_t)di.sm_count * 8;
    if (blocks > maxb) blocks = maxb;
    return (unsigned)(blocks ? blocks : 1);
}

void launch_hash_spectrum(const DeviceInfo& di, const kmer_count_pair* d_slots, uint64_t n_slots, int k, const SpecOut& o,
                          DevStatus* d_status, cudaStream_t st, int gated) {
    spectrum_scan_kernel<SPEC_HASH><<<scan_blocks(di, n_slots), 256, 0, st>>>(d_slots, n_slots, k, o, d_status, gated, 0, 1);
}

void launch_dense_spectrum(const DeviceInfo& di, const unsigned long long* d_table, int k, uint32_t rank, uint32_t n_ranks,
                           const SpecOut& o, DevStatus* d_status, cudaStream_t st) {
    const uint64_t nbins = 1ull << (2 * k);
    spectrum_scan_kernel<SPEC_DENSE><<<scan_blocks(di, nbins), 256, 0, st>>>(d_table, nbins, k, o, d_status, 0, rank, n_ranks);
}

void launch_pairs_spectrum(const DeviceInfo& di, const kmer_count_pair* d_pairs, uint64_t n, const SpecOut& o, DevStatus* d_status,
                           cudaStream_t st) {
    spectrum_scan_kernel<SPEC_PAIRS><<<scan_blocks(di, n), 256, 0, st>>>(d_pairs, n, 0, o, d_status, 0, 0, 1);
}

}  // namespace kmer
