// count_dense.cu -- K2a: GROUP BY k-mer / count(*) for small k through direct-addressed counters.
// k <= 6: 4^k uint32 bins privatised in shared memory per CTA, flushed once with 64-bit atomics.
// k <= 13: 4^k uint64 bins in HBM/L2 updated with fire-and-forget atomics (RED).
#include "kernels.cuh"

namespace kmer {

constexpr int kSmemDenseMaxK = 6;  // 4096 bins * 4 B = 16 KB

template <bool CANON = false>
__global__ void __launch_bounds__(NT) count_dense_smem_kernel(ScanArgs a, unsigned long long* __restrict__ table) {
    __shared__ ScanSmem s;
    __shared__ uint32_t bins[1 << (2 * kSmemDenseMaxK)];
    const int nbins = 1 << (2 * a.k);
    for (int b = threadIdx.x; b < nbins; b += NT) bins[b] = 0;
    TileScanner sc(a, s);  // constructor syncs
    while (sc.next()) {
#pragma unroll 4
        for (int j = 0; j < TILE / NT; j++) {
            int i = j * NT + threadIdx.x;
            if (sc.valid(i)) atomicAdd(&bins[(uint32_t)(CANON ? canon_code(sc.code(i), a.k) : sc.code(i))], 1u);
        }
        sc.release();
    }
    __syncthreads();
    for (int b = threadIdx.x; b < nbins; b += NT) {
        uint32_t c = bins[b];
        if (c) atomicAdd(&table[b], (unsigned long long)c);
    }
}

template <bool CANON = false>
__global__ void __launch_bounds__(NT) count_dense_global_kernel(ScanArgs a, unsigned long long* __restrict__ table) {
    __shared__ ScanSmem s;
    TileScanner sc(a, s);
    while (sc.next()) {
#pragma unroll 4
        for (int j = 0; j < TILE / NT; j++) {
            int i = j * NT + threadIdx.x;
            if (sc.valid(i)) atomicAdd(&table[CANON ? canon_code(sc.code(i), a.k) : sc.code(i)], 1ull);
        }
        sc.release();
    }
}

// non-zero bins -> (code,count) pairs, warp-aggregated append
__global__ void dense_compact_kernel(const unsigned long long* __restrict__ table, uint64_t nbins,
                                     kmer_count_pair* __restrict__ out, uint64_t capacity, DevStatus* status,
                                     uint32_t rank, uint32_t n_ranks) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    uint64_t nb32 = (nbins + 31) & ~31ull;
    unsigned long long total = 0;
    const int lane = threadIdx.x & 31;
    for (uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; b < nb32; b += stride) {
        unsigned long long c = (b < nbins && (n_ranks <= 1 || b % n_ranks == rank)) ? table[b] : 0;
        uint32_t m = __ballot_sync(0xffffffffu, c != 0);
        if (!m) continue;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(&status->n_distinct, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (c) {
            uint64_t idx = base + __popc(m & ((1u << lane) - 1));
            if (idx < capacity) { out[idx].code = b; out[idx].count = c; }
            else status->out_overflow = 1;
            total += c;
        }
    }
    for (int d = 16; d; d >>= 1) total += __shfl_xor_sync(0xffffffffu, total, d);
    if (lane == 0 && total) atomicAdd(&status->n_kmers, total);
}

void launch_dense_table(const DeviceInfo& di, const ScanArgs& a, unsigned long long* d_table, cudaStream_t st, bool canon) {
    uint64_t nbins = 1ull << (2 * a.k);
    cudaMemsetAsync(d_table, 0, nbins * sizeof(unsigned long long), st);
    uint64_t n_tiles = (a.n_bases + TILE - 1) / TILE;
    if (n_tiles) {
        uint64_t grid = (uint64_t)di.sm_count * 6;
        if (grid > n_tiles) grid = n_tiles;
        if (a.k <= kSmemDenseMaxK) {
            if (canon) count_dense_smem_kernel<true><<<(unsigned)grid, NT, 0, st>>>(a, d_table);
            else count_dense_smem_kernel<<<(unsigned)grid, NT, 0, st>>>(a, d_table);
        } else {
            if (canon) count_dense_global_kernel<true><<<(unsigned)grid, NT, 0, st>>>(a, d_table);
            else count_dense_global_kernel<<<(unsigned)grid, NT, 0, st>>>(a, d_table);
        }
    }
}

void launch_dense_emit(const DeviceInfo& di, const unsigned long long* d_table, int k, uint32_t rank, uint32_t n_ranks,
                       kmer_count_pair* d_pairs, uint64_t capacity, DevStatus* d_status, cudaStream_t st) {
    uint64_t nbins = 1ull << (2 * k);
    uint64_t blocks = (nbins + 255) / 256;
    uint64_t maxb = (uint64_t)di.sm_count * 8;
    if (blocks > maxb) blocks = maxb;
    dense_compact_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_table, nbins, d_pairs, capacity, d_status, rank, n_ranks);
}

void launch_count_dense(const DeviceInfo& di, const ScanArgs& a, unsigned long long* d_table, kmer_count_pair* d_pairs,
                        uint64_t capacity, cudaStream_t st, bool canon) {
    launch_dense_table(di, a, d_table, st, canon);
    launch_dense_emit(di, d_table, a.k, 0, 1, d_pairs, capacity, a.status, st);
}

}  // namespace kmer
