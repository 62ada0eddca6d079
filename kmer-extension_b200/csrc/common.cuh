// common.cuh -- device helpers shared by the k-mer kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace kmer {

constexpr int kMaxK = 32;              // MAX_KMER_LENGTH, reference kmer.h:18
constexpr uint64_t kEmpty = ~0ull;     // empty-slot sentinel of the hash tables (== 't'*32 only at k=32)
constexpr uint64_t kNoError = ~0ull;

// ---------------------------------------------------------------------------------------------
// status block shared by all kernels of one batch (device memory, mirrored to pinned host memory)
struct DevStatus {
    unsigned long long bad_char_pos;   // min flat position of a byte outside ACGTacgt (kmer.c:31-37)
    unsigned long long short_row;      // min row index with len < k               (kmer.c:310-313)
    unsigned long long n_kmers;        // windows produced
    unsigned long long n_distinct;     // groups written
    unsigned long long n_overflow;     // k-mers routed to the overflow table
    unsigned long long special_count;  // occurrences of code ~0 (k == 32 only), kept out of the tables
    unsigned long long out_overflow;   // set if an output buffer was too small
    unsigned long long pad;            // row containing bad_char_pos (resolve_bad_row_kernel)
    unsigned long long n_spill;        // partition: records that did not fit their bucket region
    unsigned long long n_failed;       // partition: buckets handed to the tier-2 kernel
    unsigned long long failed_kmers;   // k-mers (instances) in those buckets
    unsigned long long n_unique;       // split result format: k-mers written as bare codes (count 1)
    unsigned long long t2_mode;        // tier 2 of the partition counter, decided on the device: 0 not needed, 1 runs, 2 does not fit (recount)
    unsigned long long t2_slots;       // table slots tier 2 uses (a power of two, sized by what it has to count)
};

// ---------------------------------------------------------------------------------------------
// ASCII -> 2-bit SWAR encode of 4 bases (validate_sequence, kmer.c:20-41: fold case, accept acgt).
// byte 0 of w is the first base; result has the first base in bits 7..6.
// bad != 0  <=>  some byte is not one of ACGTacgt (byte-wise: nonzero byte = offending position).
__device__ __forceinline__ uint32_t enc4(uint32_t w, uint32_t& bad) {
    uint32_t x = (w >> 1) & 0x03030303u;            // A->0 C->1 G->3 T->2 (same for lower case)
    uint32_t e = x ^ ((x >> 1) & 0x01010101u);      // a=0 c=1 g=2 t=3
    uint32_t t2 = (x >> 1) & ~x & 0x01010101u;      // x == 2 (t)
    uint32_t recon = 0x61616161u + (x << 1) + t2 * 15u;  // lower-case ASCII the code stands for
    bad = (w | 0x20202020u) ^ recon;
    return (e * 0x40100401u) >> 24;
}

// 16 ASCII bytes -> one 32-bit word of 16 bases, first base in bits 31..30.
__device__ __forceinline__ uint32_t enc16(uint4 v, uint32_t& bad) {
    uint32_t b0, b1, b2, b3;
    uint32_t p = (enc4(v.x, b0) << 24) | (enc4(v.y, b1) << 16) | (enc4(v.z, b2) << 8) | enc4(v.w, b3);
    bad = b0 | b1 | b2 | b3;
    return p;
}

// index (0..15) of the first offending byte among 16, given the four per-word bad masks
__device__ __forceinline__ int first_bad_byte(uint4 v) {
    uint32_t b[4];
    enc4(v.x, b[0]); enc4(v.y, b[1]); enc4(v.z, b[2]); enc4(v.w, b[3]);
#pragma unroll
    for (int i = 0; i < 4; i++)
        if (b[i]) {
            int byte = (__ffs(b[i]) - 1) >> 3;
            return i * 4 + byte;
        }
    return 16;
}

// 64 bits of a 2-bit packed stream (uint32 words, first base in the MSBs) starting at base i
__device__ __forceinline__ uint64_t window64(const uint32_t* packed, int i) {
    int q = i >> 4, s = (i & 15) * 2;
    uint32_t w0 = packed[q], w1 = packed[q + 1], w2 = packed[q + 2];
    uint32_t hi = __funnelshift_l(w1, w0, s);
    uint32_t lo = __funnelshift_l(w2, w1, s);
    return ((uint64_t)hi << 32) | lo;
}

// bits [b, b+32) of an LSB-first bit array
__device__ __forceinline__ uint32_t bits32(const uint32_t* bits, int b) {
    int q = b >> 5, s = b & 31;
    return __funnelshift_r(bits[q], bits[q + 1], s);
}

// ---------------------------------------------------------------------------------------------
// reverse complement (canonical counting: a k-mer and its reverse complement are one group).  Codes a=0 c=1 g=2 t=3 complement
// to 3 - b = ~b, so rc is the bit-reversed complement with every 2-bit base put back in order.
__host__ __device__ __forceinline__ uint64_t brev64(uint64_t x) {
#ifdef __CUDA_ARCH__
    return __brevll(x);
#else
    x = ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
    x = ((x >> 2) & 0x3333333333333333ull) | ((x & 0x3333333333333333ull) << 2);
    x = ((x >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((x & 0x0F0F0F0F0F0F0F0Full) << 4);
    x = ((x >> 8) & 0x00FF00FF00FF00FFull) | ((x & 0x00FF00FF00FF00FFull) << 8);
    x = ((x >> 16) & 0x0000FFFF0000FFFFull) | ((x & 0x0000FFFF0000FFFFull) << 16);
    return (x >> 32) | (x << 32);
#endif
}
__host__ __device__ __forceinline__ uint32_t brev32(uint32_t x) {
#ifdef __CUDA_ARCH__
    return __brev(x);
#else
    return (uint32_t)(brev64(x) >> 32);
#endif
}
// k-mer code (first base in the high bits of the low 2k) -> code of its reverse complement
__host__ __device__ __forceinline__ uint64_t revcomp_code(uint64_t x, int k) {
    uint64_t r = brev64(~x);
    r = ((r >> 1) & 0x5555555555555555ull) | ((r & 0x5555555555555555ull) << 1);
    return r >> (64 - 2 * k);
}
// the smaller of the two codes: also the smaller of the two lower-case texts (code order is memcmp order)
__host__ __device__ __forceinline__ uint64_t canon_code(uint64_t x, int k) {
    const uint64_t r = revcomp_code(x, k);
    return r < x ? r : x;
}
// the same for the top-aligned m-mer that mmer_hash takes (its 2m top bits; the bits below are zero in the result)
__host__ __device__ __forceinline__ uint32_t revcomp_mmer(uint32_t top, int m) {
    uint32_t r = brev32(~top);
    r = ((r >> 1) & 0x55555555u) | ((r & 0x55555555u) << 1);
    return r << (32 - 2 * m);
}
__host__ __device__ __forceinline__ uint32_t canon_mmer(uint32_t top, uint32_t himask, int m) {
    const uint32_t f = top & himask, r = revcomp_mmer(top, m);
    return r < f ? r : f;
}

// ---------------------------------------------------------------------------------------------
// hashes
__device__ __host__ __forceinline__ uint64_t mix64(uint64_t x) {   // murmur3 finaliser (bijective)
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull;
    x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull;
    x ^= x >> 33;
    return x;
}
__device__ __host__ __forceinline__ uint32_t mix32(uint32_t x) {   // lowbias32 (bijective)
    x ^= x >> 16; x *= 0x7feb352du;
    x ^= x >> 15; x *= 0x846ca68bu;
    x ^= x >> 16;
    return x;
}

// Minimizer order of an m-mer: `top` holds the m-mer in its top 2m bits (himask covers them; whatever follows is masked off).
// Two multiply / xor-shift rounds INSIDE that 2m-bit field: a bijection of the 4^m m-mers onto the 4^m evenly spaced values
// i * 2^(32-2m).  Even spacing matters to the buckets below: a range of the order then holds a fixed number of m-mers, not a
// Poisson-distributed one (a plain 32-bit hash of a 26..28-bit m-mer scatters them like random points).
__device__ __forceinline__ uint32_t mmer_hash(uint32_t top, uint32_t himask, int m) {
    uint32_t t = (top & himask) * 0x9E3779B1u;              // low 32-2m bits stay zero: (x << s) * odd = ((x * odd) mod 4^m) << s
    t ^= (t >> m) & himask;
    t *= 0x85EBCA6Bu;
    t ^= (t >> (m + 1)) & himask;
    return t;
}

// Minimizer hash -> position of its bucket in [0, 2^32).  The minimizer of a window is the smallest of W (roughly independent,
// uniform) hashes, so a fraction F(u) = 1 - (1-u)^W of all windows has its minimizer at or below h = u * 2^32: small hashes
// are minimizers far more often than large ones.  Spreading the m-mers evenly over the buckets (a second hash) gives every
// bucket the same NUMBER of m-mers but very unequal loads (simulated at 41 m-mers per bucket, mean 1200 k-mers: 8 % of the
// k-mers sit in buckets above 1920).  Mapping h through F instead gives every bucket the same expected number of k-mers.
// Runs of small minimizers are long and runs of large ones short (records per k-mer grow like (1 + (W-1) u) / W), so a bucket
// of the upper end would hold several times the average number of RECORDS: the tent map 2 min(F, 1-F) pairs every slice of the
// lower half with its mirror image in the upper half, which evens out the records as well (simulated, same setting: no bucket
// above 1920 k-mers, 0.02 % of the records beyond the region capacity).  0.32 fixed point; any function of h alone keeps equal
// k-mers in one bucket.
template <int W>
__device__ __forceinline__ uint32_t bucket_position(uint32_t h) {
    const uint32_t v = ~h;                                  // 1 - u
    const uint32_t v2 = __umulhi(v, v);
    const uint32_t v4 = __umulhi(v2, v2);
    uint32_t p;                                             // (1 - u)^W
    if (W == 2) p = v2;
    else if (W == 4) p = v4;
    else if (W == 6) p = __umulhi(v4, v2);
    else {
        const uint32_t v8 = __umulhi(v4, v4);
        if (W == 8) p = v8;
        else if (W == 9) p = __umulhi(v8, v);
        else if (W == 10) p = __umulhi(v8, v2);
        else if (W == 12) p = __umulhi(v8, v4);
        else p = __umulhi(v8, v8);                          // W == 16
    }
    const uint32_t F = ~p;
    return (F ^ (uint32_t)((int32_t)F >> 31)) << 1;         // F < 1/2 ? 2F : 2(1 - F)
}
// Position -> bucket.  Single pass: bucket = position scaled to the number of buckets.  Two levels (sharded counting, two-pass
// partition: coarse partitions of F = 2^fine_shift fine buckets each): the TOP fine_shift bits of the position choose the fine
// bucket inside its coarse partition and the rest, scaled, the coarse partition -- so every coarse partition (and with it every
// owner GPU) is a comb of F narrow ranges spread evenly over the whole order, not one contiguous range: contiguous ranges
// would hold equal numbers of k-mers but, the record length depending on the position, unequal numbers of records.
__device__ __forceinline__ uint32_t coarse_bucket(uint32_t pos, uint32_t hash_buckets, int fine_shift) {
    return __umulhi(pos << fine_shift, hash_buckets >> fine_shift);
}
__device__ __forceinline__ uint32_t fine_in_coarse(uint32_t pos, int fine_shift) {
    return fine_shift ? pos >> (32 - fine_shift) : 0u;
}
// ... unless the m-mers are too coarse for that (plan.even): then they are spread by a second hash, as many per bucket everywhere
template <int W>
__device__ __forceinline__ uint32_t bucket_position(uint32_t h, int even) {
    return even ? mix32(h) : bucket_position<W>(h);
}

// ---------------------------------------------------------------------------------------------
// mbarrier + 1-D bulk async copy (TMA engine, SASS: UBLKCP) -- global -> shared staging
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// try_wait suspends the thread for a hardware time slice per call; the poll loop is bounded (2^26 polls: minutes) so that a
// copy that never arrives -- a bug, never a legal state -- traps instead of hanging the GPU.  One tight PTX loop: written in C
// the compiler unrolled it and changed the register allocation of every kernel that waits (partition_kernel +5 %).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .u32 n;\n"
        "mov.u32 n, 0;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "add.u32 n, n, 1;\n"
        "setp.lt.u32 p, n, 0x4000000;\n"
        "@p bra WAIT_LOOP;\n"
        "trap;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// bytes must be a multiple of 16; src and dst 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// the same copy with an L2 evict-first hint: for streams that are read exactly once (the dna column, a bucket's records),
// so that they do not push the partially written sectors of the scatter targets out of L2
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_g2s_stream(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

__device__ __forceinline__ uint64_t ld_nc_u64(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.global.nc.L1::no_allocate.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint4 ld_nc_u128(const void* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

}  // namespace kmer
