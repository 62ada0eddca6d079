// count_hash.cu -- K2b: GROUP BY k-mer / count(*) through an open-addressing table in HBM.
// General path for any k <= 32 and any input (also the overflow path of the minimizer-partition
// counter).  Slot = (code, count-1) in one 16-byte unit so an insert touches a single 32-byte sector;
// the table is cleared to 0xFF bytes: key 0xFF..FF = empty, stored count starts at -1.
// k == 32 uses all 64 key bits, so the one code equal to the sentinel ('t'*32) is counted in
// DevStatus::special_count instead of the table.
#include "kernels.cuh"

namespace kmer {

__device__ __forceinline__ void table_add(kmer_count_pair* slots, uint64_t mask, uint64_t code, unsigned long long cnt) {
    uint64_t h = mix64(code) & mask;
    for (;;) {
        unsigned long long prev = atomicCAS((unsigned long long*)&slots[h].code, kEmpty, code);
        if (prev == kEmpty || prev == code) {
            atomicAdd((unsigned long long*)&slots[h].count, cnt);
            return;
        }
        h = (h + 1) & mask;
    }
}

template <bool CANON = false>
__global__ void __launch_bounds__(NT) count_hash_insert_kernel(ScanArgs a, kmer_count_pair* __restrict__ slots, uint64_t mask) {
    __shared__ ScanSmem s;
    TileScanner sc(a, s);
    const int lane = threadIdx.x & 31;
    while (sc.next()) {
#pragma unroll 2
        for (int j = 0; j < TILE / NT; j++) {
            int i = j * NT + threadIdx.x;
            bool v = sc.valid(i);
            uint64_t code = sc.code(i);
            if (CANON) code = canon_code(code, a.k);       // never kEmpty: canon('t'*32) = 'a'*32
            // warp-aggregate equal keys (repetitive sequence => many equal neighbours)
            uint32_t vm = __ballot_sync(0xffffffffu, v);
            uint32_t same = __match_any_sync(0xffffffffu, code) & vm;
            if (v && lane == __ffs(same) - 1) {
                unsigned long long cnt = __popc(same);
                if (code == kEmpty) atomicAdd(&a.status->special_count, cnt);
                else table_add(slots, mask, code, cnt);
            }
        }
        sc.release();
    }
}

// merge of per-rank (k-mer, count) tables: rank `rank` adds the groups it owns (owner = hash(k-mer) % n_ranks) of a table
// that every rank sees in turn (sharded counting's exact fallback for skewed input, sharded.py).  A full table sets n_overflow.
__global__ void merge_pairs_kernel(const kmer_count_pair* __restrict__ in, uint64_t n, uint32_t rank, uint32_t n_ranks,
                                   kmer_count_pair* __restrict__ slots, uint64_t mask, DevStatus* status) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint4 raw = ld_nc_u128(&in[i]);
        const uint64_t code = ((uint64_t)raw.y << 32) | raw.x;
        const unsigned long long cnt = ((uint64_t)raw.w << 32) | raw.z;
        if (n_ranks > 1 && (uint32_t)((mix64(code ^ 0x9E3779B97F4A7C15ull) >> 32) % n_ranks) != rank) continue;
        if (code == kEmpty) { atomicAdd(&status->special_count, cnt); continue; }   // k == 32, 't'*32
        uint64_t h = mix64(code) & mask;
        bool placed = false;
        for (uint64_t tries = 0; tries <= mask; tries++) {
            const unsigned long long prev = atomicCAS((unsigned long long*)&slots[h].code, kEmpty, code);
            if (prev == kEmpty || prev == code) {
                atomicAdd((unsigned long long*)&slots[h].count, cnt);
                placed = true;
                break;
            }
            h = (h + 1) & mask;
        }
        if (!placed) atomicAdd(&status->n_overflow, cnt);
    }
}

void launch_merge_pairs(const DeviceInfo& di, const kmer_count_pair* d_in, uint64_t n, uint32_t rank, uint32_t n_ranks,
                        kmer_count_pair* d_slots, uint64_t n_slots, DevStatus* d_status, cudaStream_t st) {
    if (!n) return;
    uint64_t blocks = (n + 255) / 256;
    const uint64_t maxb = (uint64_t)di.sm_count * 8;
    if (blocks > maxb) blocks = maxb;
    merge_pairs_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_in, n, rank, n_ranks, d_slots, n_slots - 1, d_status);
}

void launch_hash_clear(kmer_count_pair* d_slots, uint64_t n_slots, cudaStream_t st) {
    cudaMemsetAsync(d_slots, 0xFF, n_slots * sizeof(kmer_count_pair), st);
}

void launch_count_hash_insert(const DeviceInfo& di, const ScanArgs& a, kmer_count_pair* d_slots, uint64_t n_slots,
                              cudaStream_t st, bool canon) {
    uint64_t n_tiles = (a.n_bases + TILE - 1) / TILE;
    if (!n_tiles) return;
    uint64_t grid = (uint64_t)di.sm_count * 6;
    if (grid > n_tiles) grid = n_tiles;
    if (canon) count_hash_insert_kernel<true><<<(unsigned)grid, NT, 0, st>>>(a, d_slots, n_slots - 1);
    else count_hash_insert_kernel<<<(unsigned)grid, NT, 0, st>>>(a, d_slots, n_slots - 1);
}

// gated != 0: the table is tier 2's and is only looked at if the device decided to run tier 2 (DevStatus::t2_mode == 1);
// the k == 32 special key is appended either way
__global__ void hash_compact_kernel(const kmer_count_pair* __restrict__ slots, uint64_t n_slots, int k,
                                    kmer_count_pair* __restrict__ out, uint64_t capacity, DevStatus* status, int gated) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    unsigned long long total = 0;
    if (gated) n_slots = status->t2_mode == 1ull ? status->t2_slots : 0;
    for (uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; b < n_slots; b += stride) {  // n_slots % 32 == 0
        uint4 raw = ld_nc_u128(&slots[b]);
        uint64_t code = ((uint64_t)raw.y << 32) | raw.x;
        uint64_t cnt = (((uint64_t)raw.w << 32) | raw.z) + 1;
        bool occ = code != kEmpty;
        uint32_t m = __ballot_sync(0xffffffffu, occ);
        if (!m) continue;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(&status->n_distinct, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (occ) {
            uint64_t idx = base + __popc(m & ((1u << lane) - 1));
            if (idx < capacity) { out[idx].code = code; out[idx].count = cnt; }
            else status->out_overflow = 1;
            total += cnt;
        }
    }
    for (int d = 16; d; d >>= 1) total += __shfl_xor_sync(0xffffffffu, total, d);
    if (lane == 0 && total) atomicAdd(&status->n_kmers, total);
    // the one key that cannot live in the table (k == 32, 't'*32)
    if (blockIdx.x == 0 && threadIdx.x == 0 && k == 32) {
        unsigned long long sc = status->special_count;
        if (sc) {
            unsigned long long idx = atomicAdd(&status->n_distinct, 1ull);
            if (idx < capacity) { out[idx].code = kEmpty; out[idx].count = sc; }
            else status->out_overflow = 1;
            atomicAdd(&status->n_kmers, sc);
        }
    }
}

void launch_hash_compact(const DeviceInfo& di, const kmer_count_pair* d_slots, uint64_t n_slots, int k,
                         kmer_count_pair* d_pairs, uint64_t capacity, DevStatus* d_status, cudaStream_t st, int gated) {
    uint64_t blocks = (n_slots + 255) / 256;
    uint64_t maxb = (uint64_t)di.sm_count * 8;
    if (blocks > maxb) blocks = maxb;
    hash_compact_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_slots, n_slots, k, d_pairs, capacity, d_status, gated);
}

}  // namespace kmer
