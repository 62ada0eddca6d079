// count_part.cu -- K2c: GROUP BY k-mer / count(*) for 14 <= k <= 32 by minimizer partitioning.
//
// HBM cannot afford one random 32-byte sector per k-mer (what a global hash table costs), and the
// SMs cannot afford one atomic per k-mer in the partitioning pass.  So the column is regrouped in
// two kernels with a compact intermediate:
//
//  partition_kernel   tile scanner (TMA-staged ASCII -> 2-bit) -> for every window the minimum
//                     hashed m-mer over its W m-mers -> bucket = mix(min) * NB >> 32.
//                     Identical k-mers have identical minimizers, hence the same bucket.
//                     Consecutive windows that share a minimizer are emitted as ONE super-k-mer record
//                     (2 bits per base + a length), appended to the bucket's region with a single
//                     64-bit atomicAdd per record (about 0.22 records per k-mer at W = 8).
//  bucket_count_kernel one CTA per bucket (about 1200 k-mers): a bitmap filter proves most k-mers unique
//                     (they are written straight to the result), the rest is counted exactly in a
//                     2048-slot shared-memory hash table (64-bit atomicCAS).
//  refine_*_kernel    sharded counting only: a source GPU partitions into few coarse partitions, the owner
//                     splits them into the fine buckets above.
//
// HBM traffic: read N bases once, write + read ~1.8 B per k-mer of records, write 16 B per group.
//
// What does not fit is handled in tiers (skewed / repetitive input):
//   tier 2  a bucket whose region overflowed (extra records go to a spill list) or that holds more
//           k-mers than the leaf takes (2047) is put on a failed list and emits nothing; one more
//           kernel counts exactly those buckets' records in a global hash table and appends them;
//   tier 3  if even the spill list overflows, DevStatus::n_overflow is set and the caller recounts
//           the whole batch with the global-hash-table path (count_hash.cu).
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "spectrum.cuh"

namespace kmer {

constexpr int LEAF_SLOTS = 1024;          // shared-memory table slots per bucket (exact counts of the repeated k-mers)
#ifndef LEAF_THREADS_N
#define LEAF_THREADS_N 128
#endif
constexpr int LEAF_THREADS = LEAF_THREADS_N;
constexpr uint32_t TARGET_KMERS_PER_BUCKET = 1200;   // about half of what a bucket may hold; the tail is handled by tier 2

// ---------------------------------------------------------------------------------------------
// record formats
//   RECW == 1 (k <= 26): one uint64 : bases 0..29 in bits 63..4 (first base highest), (L-1) in bits 3..0
//   RECW == 2 (k >= 27): two uint64 : hi = bases 0..31 ; lo = bases 32..60 in bits 63..6, (L-1) in bits 5..0
// L = number of k-mers of the record (1..16), which covers L+k-1 bases.

template <int RECW>
struct Rec;
template <>
struct Rec<1> {
    uint64_t v;
};
template <>
struct alignas(16) Rec<2> {
    uint64_t hi, lo;
};

// ---------------------------------------------------------------------------------------------
// partition

#ifndef PART_MINB
#define PART_MINB 3
#endif
// CANON: canonical counting needs a k-mer and its reverse complement in one bucket, so the minimizer is strand-symmetric: the
// hashed m-mer is the canonical one (min(m-mer, rc)), and the W m-mers of a window sit symmetrically in it, offset by
// (k - m - W + 1) / 2 bases (make_partition_plan keeps that even).  Then a k-mer and its reverse complement hash the same set of
// canonical m-mers.  The records still carry the forward bases.
template <int W, int RECW, bool CANON = false>
__global__ void __launch_bounds__(NT, PART_MINB) partition_kernel(ScanArgs a, PartitionPlan plan, unsigned long long* __restrict__ fill,
                                                       Rec<RECW>* __restrict__ recs, Rec<RECW>* __restrict__ spill) {
    __shared__ ScanSmem s;
    __shared__ unsigned long long runs[TILE];   // (minimizer hash << 32) | (windows << 16) | tile-relative start base
    __shared__ uint32_t bdm[TILE / 32 + 2];     // bit p: a run cannot continue through window p (run start or invalid window)
    TileScanner sc(a, s);
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int k = a.k;
    const int m = plan.m;
    const uint32_t rmax = plan.rmax;
    const uint32_t himask = 0xffffffffu << (32 - 2 * m);
    unsigned long long overflow_kmers = 0;
    if (t < 2) bdm[TILE / 32 + t] = 0xffffffffu;   // the tile end ends every run
    uint64_t pol_last, pol_first;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_last));
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_first));

    // one super-k-mer record: L windows starting at tile-relative base p go to bucket b
    auto put_record = [&](uint32_t b, uint32_t slot, int p, int L) {
        const int c = p >> 4, sh = 2 * (p & 15);
        const uint32_t w0 = s.packed[c], w1 = s.packed[c + 1], w2 = s.packed[c + 2], w3 = s.packed[c + 3];
        const uint32_t r0w = __funnelshift_l(w1, w0, sh), r1w = __funnelshift_l(w2, w1, sh), r2w = __funnelshift_l(w3, w2, sh);
        const int nb = L + k - 1;                                  // bases covered
        Rec<RECW>* dst = nullptr;
        if (slot < plan.cap) dst = recs + ((uint64_t)b * plan.cap + slot);
        else {                                                      // region full: spill list (tier 2), else recount
            unsigned long long si = atomicAdd(&a.status->n_spill, 1ull);
            if (si < plan.spill_cap) dst = spill + si;
            else overflow_kmers += L;
        }
        if (dst) {
            if (RECW == 1) {
                uint64_t v = ((uint64_t)r0w << 32) | r1w;
                v &= ~0ull << (64 - 2 * nb);                       // nb <= 30
                // a region's last, partially written 32-byte sector must stay in L2 until it is complete (else every
                // record costs a sector fill from HBM): evict-last while it fills up, evict-first with its fourth record
                const uint64_t pol = (slot & 3u) == 3u ? pol_first : pol_last;
                asm volatile("st.global.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(dst), "l"(v | (uint64_t)(L - 1)), "l"(pol) : "memory");
            } else {
                uint64_t hi = ((uint64_t)r0w << 32) | r1w;
                uint64_t lo = (uint64_t)r2w << 32;                  // bases 32..47 (nb <= 47)
                if (nb <= 32) { hi &= ~0ull << (64 - 2 * nb); lo = 0; }
                else lo &= ~0ull << (128 - 2 * nb);
                const uint64_t pol = (slot & 1u) ? pol_first : pol_last;
                asm volatile("st.global.L2::cache_hint.v2.u64 [%0], {%1, %2}, %3;" ::"l"(dst), "l"(hi), "l"(lo | (uint64_t)(L - 1)), "l"(pol)
                             : "memory");
            }
        }
    };

    while (sc.next()) {
        const uint32_t* bnd = sc.bnd();
        // this thread's 16 windows start at tile-relative bases 16t .. 16t+15 and need bases up to 16t+46;
        // window 16t-1 (the previous thread's last) is looked at as well, so that runs continue across threads
        uint32_t w[3];
        w[0] = s.packed[t]; w[1] = s.packed[t + 1]; w[2] = s.packed[t + 2];
        uint32_t wm1 = t ? s.packed[t - 1] : 0u;
        if (CANON) {                                                  // the m-mers of window j start at base j + off
            const int sh = k - m - W + 1;                             // 2 * off: off <= 5, so j + off <= 31 below
            const uint32_t w3 = s.packed[t + 3];
            wm1 = __funnelshift_l(w[0], wm1, sh);
            w[0] = __funnelshift_l(w[1], w[0], sh);
            w[1] = __funnelshift_l(w[2], w[1], sh);
            w[2] = __funnelshift_l(w3, w[2], sh);
        }
        // validity of the windows: no row start in (i, i+k-1], and inside the input
        uint32_t vmask = 0;      // bit j+1: window j is valid (j = -1 .. 15)
        {
            const int b0 = 16 * t;                                   // bit q of bw: a row starts at base 16t + q
            const uint32_t lo = bits32(bnd, b0), hi = bits32(bnd, b0 + 32);
            const uint64_t bw = ((uint64_t)hi << 32) | lo;
            const uint64_t remaining = a.n_bases > sc.t0 + 16ull * t ? a.n_bases - (sc.t0 + 16ull * t) : 0;
            if (remaining >= 16 && ((bw >> 1) & ((1ull << (15 + k - 1)) - 1ull)) == 0) vmask = 0x1fffeu;   // the common case
            else {
#pragma unroll
                for (int j = 0; j < 16; j++) {
                    bool ok = (((uint32_t)(bw >> (j + 1)) & sc.kmask) == 0) && ((uint64_t)j < remaining);
                    vmask |= (uint32_t)ok << (j + 1);
                }
            }
            if (t && remaining && (lo & sc.kmask) == 0) vmask |= 1u;  // window 16t-1: bits 16t .. 16t+k-2
        }
        uint32_t starts = 0;
        uint32_t h[17 + W - 1];                                       // h[j+1]: minimizer hash of window j
        if (vmask >> 1) {
            // hashed m-mers at bases -1 .. 15+W-1 of this chunk
#pragma unroll
            for (int j = -1; j < 16 + W - 1; j++) {
                uint32_t top;                                         // 16 bases starting at base j
                if (j < 0) top = __funnelshift_l(w[0], wm1, 30);
                else {
                    const int q = j >> 4, sh = (j & 15) * 2;
                    top = __funnelshift_l(w[q + 1], w[q], sh);
                }
                h[j + 1] = mmer_hash(CANON ? canon_mmer(top, himask, m) : top, himask, m);
            }
            // sliding minimum over W consecutive m-mers: log-steps up to the largest power of two P <= W, then two
            // overlapping P-windows cover a W-window
            constexpr int P = W >= 16 ? 16 : (W >= 8 ? 8 : (W >= 4 ? 4 : 2));
#pragma unroll
            for (int step = 1; step < P; step <<= 1) {
#pragma unroll
                for (int j = 0; j < 17 + W - 1 - step; j++) h[j] = min(h[j], h[j + step]);
            }
            if (W > P) {
#pragma unroll
                for (int j = 0; j < 17; j++) h[j] = min(h[j], h[j + W - P]);
            }
            // a run starts where the minimizer changes (identical k-mers have identical minimizers, hence the same
            // bucket = mix(minimizer hash); the bucket itself is only computed once per run, at emission)
#pragma unroll
            for (int j = 0; j < 16; j++) {
                const bool v = (vmask >> (j + 1)) & 1u, pv = (vmask >> j) & 1u;
                starts |= (uint32_t)(v && (!pv || h[j + 1] != h[j])) << j;
            }
        }
        // A run is emitted by ONE lane, piece by piece: keep it short.  It may run on from the previous thread's chunk only if
        // it began there, and never across a warp edge -- so a homopolymer costs every lane one short run, not one lane thousands.
        {
            const uint32_t prev_starts = __shfl_up_sync(0xffffffffu, starts, 1);
            if (((vmask >> 1) & 1u) && (lane == 0 || prev_starts == 0)) starts |= 1u;
        }
        const uint32_t bd = (starts | ~(vmask >> 1)) & 0xffffu;
        reinterpret_cast<uint16_t*>(bdm)[t] = (uint16_t)bd;
        // ---- the warp's runs, compacted into the warp's own list (warp-wide exclusive scan of the run counts)
        const uint32_t nrun = __popc(starts);
        uint32_t incl = nrun;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += n;
        }
        const uint32_t n_warp_runs = __shfl_sync(0xffffffffu, incl, 31);
        unsigned long long* wruns = runs + warp * 512;
        if (starts) {
            uint32_t rbase = incl - nrun;
#pragma unroll
            for (int j = 0; j < 16; j++)
                if ((starts >> j) & 1u) wruns[rbase++] = ((unsigned long long)h[j + 1] << 32) | (uint32_t)(16 * t + j);
        }
        // ---- emission: run i of the warp is handled by lane i % 32.  A run never leaves its warp's 512 windows (lane 0 always
        //      starts one), so its length follows from the warp's OWN boundary bits: no tile barrier, and ONE 64-bit atomicAdd
        //      per record on the bucket's fill word -- record count in the low half (the returned value is the region slot),
        //      k-mer count in the high half.  Up to EMIT_Q round trips per lane are in flight.
        constexpr int EMIT_Q = 6;
        __syncwarp();
        auto run_length = [&](uint32_t p0) {                          // the run ends before the next boundary bit after its first window
            const uint32_t wend = (p0 | 511u) + 1u;                   // ... or with the warp's windows
            uint32_t p = p0 + 1, R = 1;
            while (p < wend) {
                uint32_t nb32 = bits32(bdm, p);
                const uint32_t rem = wend - p;
                if (rem < 32) nb32 |= 0xffffffffu << rem;             // bits past the warp's end belong to another warp
                if (nb32) { R += __ffs(nb32) - 1; break; }
                R += 32; p += 32;
            }
            return R;
        };
        uint32_t posq[EMIT_Q], bq[EMIT_Q], slot[EMIT_Q];             // run length << 16 | start base ; bucket ; region slot
#pragma unroll
        for (int q = 0; q < EMIT_Q; q++) {
            const uint32_t r = q * 32 + lane;
            posq[q] = 0xffffffffu; bq[q] = 0; slot[q] = 0;
            if (r < n_warp_runs) {
                const unsigned long long d = wruns[r];
                bq[q] = coarse_bucket(bucket_position<W>((uint32_t)(d >> 32), plan.even), plan.hash_buckets, plan.fine_shift);
                const uint32_t R = run_length((uint32_t)d);
                posq[q] = (uint32_t)d | (R << 16);
                const uint32_t L0 = R < rmax ? R : rmax;
                slot[q] = (uint32_t)atomicAdd(&fill[bq[q]], ((unsigned long long)L0 << 32) | 1ull);
            }
        }
        // one run: its first record takes the slot reserved above; a run longer than one record holds takes further slots
        // (repetitive text)
        auto emit_run = [&](uint32_t b, uint32_t slot0, uint32_t p0, uint32_t R) {
            const uint32_t L0 = R < rmax ? R : rmax;
            put_record(b, slot0, (int)p0, (int)L0);
            for (uint32_t off = rmax; off < R; off += rmax) {
                const uint32_t L = R - off < rmax ? R - off : rmax;
                const unsigned long long o2 = atomicAdd(&fill[b], ((unsigned long long)L << 32) | 1ull);
                put_record(b, (uint32_t)o2, (int)(p0 + off), (int)L);
            }
        };
#pragma unroll
        for (int q = 0; q < EMIT_Q; q++)
            if (posq[q] != 0xffffffffu) emit_run(bq[q], slot[q], posq[q] & 0xffffu, posq[q] >> 16);
        for (uint32_t r = EMIT_Q * 32 + lane; r < n_warp_runs; r += 32) {   // more than 192 runs in 512 windows: rare
            const unsigned long long d = wruns[r];
            const uint32_t b = coarse_bucket(bucket_position<W>((uint32_t)(d >> 32), plan.even), plan.hash_buckets, plan.fine_shift);
            const uint32_t R = run_length((uint32_t)d);
            const uint32_t L0 = R < rmax ? R : rmax;
            const uint32_t s0 = (uint32_t)atomicAdd(&fill[b], ((unsigned long long)L0 << 32) | 1ull);
            emit_run(b, s0, (uint32_t)d, R);
        }
        sc.release();
    }
    if (overflow_kmers) atomicAdd(&a.status->n_overflow, overflow_kmers);
}

// ---------------------------------------------------------------------------------------------
// per-bucket counting
//
// One CTA (128 threads) per bucket (about 1200 k-mers, at most LEAF_MAX_KMERS).  Most k-mers of a bucket occur once;
// proving that is much cheaper than inserting them into an exact table, so the table only sees the rest:
//   stage   : the bucket's record region (contiguous in HBM) is brought to shared memory by the TMA engine
//             (cp.async.bulk + mbarrier), double buffered: the copy for bucket i+1 runs behind bucket i.
//   index   : thread t takes the records [t*c, t*c+c) (c = ceil(records / 128)); a warp-wide prefix sum of their lengths
//             numbers the bucket's k-mers ("key index").  Every warp owns a range of key indices that starts on a multiple
//             of 32 (one shared atomicAdd per warp hands it out), so a 32-key block never mixes two warps' records.
//             Per record the first key index goes to P[], a start bit to a bit mask over the key indices, and the record
//             that covers the first key of a 32-key block to blk[].                               -- barrier (E) --
//   mark    : thread t owns key indices t, t+128, ...: all lanes of a warp look at the SAME 32-key block, so
//             record(i) = blk[block] + popc(start bits of the block up to the lane) -- one POPC, two broadcast loads --
//             and the k-mer is two shifts of that record.  No per-k-mer array exists in shared memory: the keys live in
//             REGISTERS from here to the emission, every lane busy whatever the record lengths are.  Each k-mer sets bit
//             hash(k-mer) of bitmap A (atom.or with return); whoever finds the bit already set sets the same bit of
//             bitmap B.                                                                          -- barrier (M) --
//   classify: a k-mer whose B bit is clear is the ONLY k-mer of the bucket in its cell: it is unique, count 1.
//             The others (true repeats and the ~4 % that merely share a cell) put their key index on the "slow list".
//                                                                                                -- barrier (L) --
//   count   : the slow list is spread evenly over the warps and counted exactly in a 1024-slot open-addressing
//             table: one 64-bit shared atomicCAS per lane per iteration (double hashing); a lane whose key is placed
//             or found takes the warp's next k-mer (ballot + popc on a warp-uniform cursor: no atomics, no idle
//             lanes).  k <= 26: the count lives in the 12 spare top bits of the key word; k >= 27: separate 32-bit
//             counters.  The slots a warp claims are listed in place of its consumed slow-list entries.  A key that
//             finds the table full (more than 1023 distinct repeated k-mers in one bucket) is handed to tier 2 as a
//             one-k-mer spill record.                                                            -- barrier (B) --
//   emit    : unique k-mers straight from the registers, table entries from the claimed-slot lists (which also
//             resets the table); both as coalesced 16-byte (k-mer, count) pairs (or bare codes in the split format).
//             Output ranges: one global atomicAdd per bucket for the unique k-mers, one per warp that claimed slots.
//   SPEC    : the spectrum result format (count of counts, spectrum.cuh) instead of the groups: the unique k-mers are only
//             counted (a register per warp, added to the CTA's bin 1 at the end), table entries are binned in the CTA's shared
//             histogram (counts < 64), into hist[] (counts < hist_len) or appended to the tail; no output range is handed out
//             and nothing is stored per group.  out / capacity are the tail, out_u / capacity_u the histogram and its length.
// Buckets above LEAF_MAX_KMERS, or whose region overflowed in the partition pass, go to tier 2 up front.
// Shared memory is addressed through explicit 32-bit shared addresses (ld/st/atom.shared PTX).

constexpr int LEAF_KPT = 16;                                          // key indices per thread
constexpr uint32_t LEAF_KEYS = LEAF_KPT * LEAF_THREADS;              // 2048 key indices
constexpr int LEAF_WARPS = LEAF_THREADS / 32;
constexpr uint32_t LEAF_MAX_KMERS = LEAF_KEYS - 32 * LEAF_WARPS;     // 1920: every warp's index range is padded to 32
constexpr int LEAF_CELLS = 32768;                                    // bits per filter bitmap
constexpr int LEAF_BLOCKS = LEAF_KEYS / 32;                          // 32-key blocks
#ifndef LEAF_MINB
#define LEAF_MINB 7
#endif

__device__ __forceinline__ unsigned long long atoms_cas64(uint32_t a, unsigned long long cmp, unsigned long long val) {
    unsigned long long old;
    asm volatile("atom.shared.cas.b64 %0, [%1], %2, %3;" : "=l"(old) : "r"(a), "l"(cmp), "l"(val) : "memory");
    return old;
}
__device__ __forceinline__ uint32_t atoms_add32(uint32_t a, uint32_t v) {
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
    return old;
}
__device__ __forceinline__ uint32_t atoms_or32(uint32_t a, uint32_t v) {
    uint32_t old;
    asm volatile("atom.shared.or.b32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
    return old;
}
__device__ __forceinline__ void reds_or32(uint32_t a, uint32_t v) {
    asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void reds_add32(uint32_t a, uint32_t v) {
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void reds_add64(uint32_t a, unsigned long long v) {
    asm volatile("red.shared.add.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory");
}
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long lds64(uint32_t a) {
    unsigned long long v;
    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t lds16(uint32_t a) {
    uint16_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts16(uint32_t a, uint32_t v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((uint16_t)v) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t a, unsigned long long v) {
    asm volatile("st.shared.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory");
}
__device__ __forceinline__ void lds128(uint32_t a, unsigned long long& x, unsigned long long& y) {
    asm volatile("ld.shared.v2.u64 {%0,%1}, [%2];" : "=l"(x), "=l"(y) : "r"(a) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void mbar_wait_s(uint32_t bar, uint32_t parity) {   // bounded like mbar_wait (common.cuh)
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .u32 n;\n"
        "mov.u32 n, 0;\n"
        "LEAF_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LEAF_DONE;\n"
        "add.u32 n, n, 1;\n"
        "setp.lt.u32 p, n, 0x4000000;\n"
        "@p bra LEAF_WAIT;\n"
        "trap;\n"
        "LEAF_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}

// cell of the filter bitmaps (15 bits) and, decorrelated from it, the slot hash of the exact table
__device__ __forceinline__ uint32_t leaf_mix(uint64_t key) {
    return (uint32_t)key * 0x9E3779B1u + (uint32_t)(key >> 32) * 0x85EBCA6Bu;
}
// cell of the filter bitmaps (15 bits).  Both halves of the key must go in: hashing the low word alone is one IMAD cheaper but
// sends 2x as many k-mers to the exact table (measured: 7.0 instead of 6.45 ms for the 1 GB bench)
__device__ __forceinline__ uint32_t leaf_cell(uint64_t key) { return leaf_mix(key) >> 17; }

struct BucketInfo {
    uint32_t nrec, nk;
    bool overflow;
    __device__ __forceinline__ bool usable() const { return nrec != 0 && !overflow && nk <= LEAF_MAX_KMERS; }
};

__device__ __forceinline__ BucketInfo bucket_info(const unsigned long long* __restrict__ fill, const PartitionPlan& plan, uint32_t b) {
    BucketInfo bi;
    const unsigned long long f = fill[b];
    bi.nrec = (uint32_t)f;
    bi.nk = (uint32_t)(f >> 32);
    bi.overflow = (uint32_t)f > plan.cap;
    return bi;
}

template <int RECW, bool SPLIT, bool SPEC = false, bool CANON = false>
__global__ void __launch_bounds__(LEAF_THREADS, LEAF_MINB) bucket_count_kernel(PartitionPlan plan, int k,
                                                                       const unsigned long long* __restrict__ fill,
                                                                       const Rec<RECW>* __restrict__ recs,
                                                                       kmer_count_pair* __restrict__ out, uint64_t capacity,
                                                                       uint64_t* __restrict__ out_u, uint64_t capacity_u,
                                                                       uint32_t* __restrict__ failed_ids, Rec<RECW>* __restrict__ spill,
                                                                       DevStatus* status, uint32_t bucket_begin, uint32_t bucket_end) {
    constexpr bool PACKED = RECW == 1;                        // count in bits 63..52 of the key word (k <= 26)
    constexpr uint32_t RECB = RECW * 8;
    constexpr uint64_t KEYMASK = PACKED ? ((1ull << 52) - 1ull) : ~0ull;
    extern __shared__ __align__(16) unsigned char leaf_dyn[];
    uint32_t tbl_s = smem_u32(leaf_dyn);                                       // u64[LEAF_SLOTS]
    asm volatile("" : "+r"(tbl_s));                                            // keep it in a register (no rematerialisation)
    const uint32_t cnt_s = tbl_s + LEAF_SLOTS * 8;                             // u32[LEAF_SLOTS]   (k >= 27 only)
    const uint32_t bma_s = cnt_s + (PACKED ? 0 : LEAF_SLOTS * 4);             // bitmap A
    const uint32_t bmb_s = bma_s + LEAF_CELLS / 8;                             // bitmap B
    const uint32_t slow_s = bmb_s + LEAF_CELLS / 8;                            // u16[LEAF_KEYS]: slow list (key indices), then claimed slots
    const uint32_t p_s = slow_s + LEAF_KEYS * 2;                               // u16[cap + 2]: first key index of every record
    const uint32_t rec0_s = p_s + ((((uint32_t)plan.cap + 2u) * 2u + 15u) & ~15u);   // staged records, two buffers
    const uint32_t rec_stride = (((uint32_t)plan.cap + 2u) * RECB + 15u) & ~15u;
    const uint32_t hist_s = rec0_s + 2u * rec_stride;                          // SPEC: u32[SPEC_SBINS]
    __shared__ __align__(8) uint64_t s_mbar;
    __shared__ uint32_t s_mask[2][LEAF_BLOCKS];                                // per bucket parity: bit i&31 of word i>>5: a record starts at key index i
    __shared__ uint32_t s_blk[LEAF_BLOCKS];                                    // record that covers key index 32*block
    __shared__ uint32_t s_kcur;                                                // index phase: next free key index (a multiple of 32)
    __shared__ uint32_t s_nuniq[2], s_nslow[2];                                // per bucket parity
    __shared__ unsigned long long s_obase[2];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const uint32_t lane_lt = (1u << lane) - 1u;
    const uint32_t lane_starts = (2u << lane) - 2u;                            // start bits 1..lane of a 32-key block
    const int kshift = 64 - 2 * k;
    const uint32_t mbar_s = smem_u32(&s_mbar);
    const uint32_t kcur_s = smem_u32(&s_kcur);
    const uint32_t blk_s = smem_u32(s_blk);
    unsigned long long special_total = 0, kmers_total = 0;
    for (int i = t; i < LEAF_SLOTS / 2; i += LEAF_THREADS) sts128(tbl_s + 16 * i, ~0u, ~0u, ~0u, ~0u);
    if (!PACKED)
        for (int i = t; i < LEAF_SLOTS / 4; i += LEAF_THREADS) sts128(cnt_s + 16 * i, 0u, 0u, 0u, 0u);
    for (int i = t; i < 2 * LEAF_CELLS / 128; i += LEAF_THREADS) sts128(bma_s + 16 * i, 0u, 0u, 0u, 0u);   // A and B
    if (t < LEAF_BLOCKS) { s_mask[0][t] = 0; s_mask[1][t] = 0; }
    if (t < 2) { s_nuniq[t] = 0; s_nslow[t] = 0; }
    if (t == 0) { s_kcur = 0; mbar_init(&s_mbar, 1); mbar_fence_init(); }
    if (SPEC)
        for (int i = t; i < SPEC_SBINS; i += LEAF_THREADS) sts32(hist_s + 4 * i, 0u);
    uint32_t uniq_total = 0;                                            // SPEC: unique k-mers of this warp (the same on every lane)
    __syncthreads();

    // thread 0: start the bulk copy of bucket b's records (padded to 16 bytes; read once: L2 evict-first)
    const uint64_t pol_stream = l2_evict_first_policy();
    auto issue = [&](uint32_t b, uint32_t buf) {
        const uint32_t n = (uint32_t)fill[b];
        const uint32_t nb = (n * RECB + 15u) & ~15u;
        mbar_arrive_expect_tx(&s_mbar, nb);
        if (nb)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                             rec0_s + buf * rec_stride),
                         "l"(recs + (uint64_t)b * plan.cap), "r"(nb), "r"(mbar_s), "l"(pol_stream)
                         : "memory");
    };

    uint32_t par = 0, phase = 0, rb = 0;                                // bucket parity, mbarrier phase, record buffer
    BucketInfo cur;
    cur.nrec = 0; cur.nk = 0; cur.overflow = false;
    const uint32_t b_first = bucket_begin + blockIdx.x;
    if (b_first < bucket_end) cur = bucket_info(fill, plan, b_first);
    if (t == 0 && cur.usable()) issue(b_first, 0);

    for (uint32_t b = b_first; b < bucket_end; b += gridDim.x) {
        const uint32_t b_next = b + gridDim.x;
        BucketInfo nxt;
        nxt.nrec = 0; nxt.nk = 0; nxt.overflow = false;
        if (b_next < bucket_end) nxt = bucket_info(fill, plan, b_next);   // in flight during the index phase
        if (!cur.usable()) {                                            // uniform across the CTA
            if (t == 0) {
                if (cur.nrec) {                                         // does not fit on chip: tier 2
                    uint32_t idx = (uint32_t)atomicAdd(&status->n_failed, 1ull);
                    failed_ids[idx] = b;
                    atomicAdd(&status->failed_kmers, (unsigned long long)cur.nk);
                }
                if (nxt.usable()) issue(b_next, rb);                    // nothing is staged for this bucket
            }
            cur = nxt;
            continue;
        }
        mbar_wait_s(mbar_s, phase);
        phase ^= 1u;
        const uint32_t rec_s = rec0_s + rb * rec_stride;
        const uint32_t mask_s = smem_u32(s_mask[par]);
        auto rec_len = [&](uint32_t r) -> uint32_t {
            return RECW == 1 ? (lds32(rec_s + 8 * r) & 15u) + 1 : (lds32(rec_s + 16 * r + 8) & 63u) + 1;
        };
        // window j of record r (the low length bits are shifted out: j + k <= 30 resp. 61 bases)
        auto window = [&](uint32_t r, uint32_t j) -> uint64_t {
            if (RECW == 1) return (lds64(rec_s + 8 * r) << (2 * j)) >> kshift;
            unsigned long long hi, lo;
            lds128(rec_s + 16 * r, hi, lo);
            return (j ? ((hi << (2 * j)) | (lo >> (64 - 2 * j))) : hi) >> kshift;
        };
        // CANON: every key is the canonical code of its window, formed where mark and count read it.  A record may then hold
        // both x and rc(x): nothing below assumes the keys of a record are distinct.
        // ---- index: thread t numbers the k-mers of records [t*c, t*c + c)
        const uint32_t nrec = cur.nrec;
        {
            const uint32_t c = (nrec + LEAF_THREADS - 1) / LEAF_THREADS;
            const uint32_t r0 = t * c, r1 = min(r0 + c, nrec);
            uint32_t S = 0;
            for (uint32_t r = r0; r < r1; r++) S += rec_len(r);
            uint32_t incl = S;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += n;
            }
            uint32_t base = 0;
            if (lane == 31 && incl) base = atoms_add32(kcur_s, (incl + 31u) & ~31u);   // the warp's index range starts on a 32-key block
            base = __shfl_sync(0xffffffffu, base, 31);
            uint32_t p = base + incl - S;
            for (uint32_t r = r0; r < r1; r++) {
                const uint32_t L = rec_len(r), e = p + L - 1;
                sts16(p_s + 2 * r, p);
                reds_or32(mask_s + 4 * (p >> 5), 1u << (p & 31u));
                if ((p & 31u) == 0 || (e >> 5) != (p >> 5)) sts32(blk_s + 4 * (e >> 5), r);   // covers the first key of block e>>5
                p += L;
            }
        }
        __syncthreads();                                                // (E) index complete; the other record buffer is free
        const uint32_t nkeys = s_kcur;                                  // key indices handed out (padded per warp)
        if (t == 0 && nxt.usable()) issue(b_next, rb ^ 1u);
        // ---- mark: thread t owns key indices t, t+128, ...  (block = warp + 4 i, bit = lane)
        uint64_t key[LEAF_KPT];
        uint32_t valid = 0, multi = 0, special = 0;                     // bit i: key i exists / shares its cell
#pragma unroll
        for (int i = 0; i < LEAF_KPT; i++) {
            key[i] = 0;
            if (i * LEAF_THREADS >= (int)nkeys) break;                  // uniform
            const uint32_t blk = warp + LEAF_WARPS * i;
            if (blk * 32u >= nkeys) break;                              // uniform per warp: the block was not handed out
            const uint32_t r = lds32(blk_s + 4 * blk) + __popc(lds32(mask_s + 4 * blk) & lane_starts);
            const uint32_t j = (uint32_t)(t + i * LEAF_THREADS) - lds16(p_s + 2 * r);
            if (j < rec_len(r)) {                                       // not in the padding behind the warp's last record
                key[i] = window(r, j);
                if (CANON) key[i] = canon_code(key[i], k);
                if (RECW == 2 && key[i] == kEmpty) special++;           // k == 32, 't'*32: kept out of the tables
                else {
                    valid |= 1u << i;
                    const uint32_t cell = leaf_cell(key[i]);
                    const uint32_t bit = 1u << (cell & 31u), w = (cell >> 5) * 4;
                    if (atoms_or32(bma_s + w, bit) & bit) {
                        reds_or32(bmb_s + w, bit);
                        multi |= 1u << i;
                    }
                }
            }
        }
        __syncthreads();                                                // (M) both bitmaps final
        if (t == 0) s_kcur = 0;
        // ---- classify: unique k-mers stay in their registers, the others put their key index on the slow list
#pragma unroll
        for (int i = 0; i < LEAF_KPT; i++) {
            if (i * LEAF_THREADS >= (int)nkeys) break;
            if ((valid >> i) & 1u) {
                bool slow = (multi >> i) & 1u;
                if (!slow) {
                    const uint32_t cell = leaf_cell(key[i]);
                    slow = (lds32(bmb_s + (cell >> 5) * 4) >> (cell & 31u)) & 1u;
                }
                if (slow) {
                    multi |= 1u << i;
                    sts16(slow_s + 2 * atoms_add32(smem_u32(&s_nslow[par]), 1u), t + i * LEAF_THREADS);
                }
            }
        }
        const uint32_t uniq = valid & ~multi;
        // the warp's unique k-mers get a contiguous share of the bucket's output
        const uint32_t wuniq = __reduce_add_sync(0xffffffffu, (uint32_t)__popc(uniq));
        uint32_t woff = 0;
        if (SPEC) uniq_total += wuniq;
        else {
            if (lane == 0 && wuniq) woff = atoms_add32(smem_u32(&s_nuniq[par]), wuniq);
            woff = __shfl_sync(0xffffffffu, woff, 0);
        }
        __syncthreads();                                                // (L) slow list complete
        const uint32_t ns = s_nslow[par];
        unsigned long long ubase = 0;
        if (t == 0 && !SPEC) {
            const uint32_t nu = s_nuniq[par];
            if (nu) ubase = atomicAdd(SPLIT ? &status->n_unique : &status->n_distinct, (unsigned long long)nu);   // consumed after the next barrier
        }
        // both bitmaps are dead: clear them for the next bucket
        for (int i = t; i < 2 * LEAF_CELLS / 128; i += LEAF_THREADS) sts128(bma_s + 16 * i, 0u, 0u, 0u, 0u);
        // ---- count: the slow list is cut into one slice per warp, but never thinner than 32 entries (a warp pays for
        //      the probe loop whether 1 or 32 of its lanes are busy)
        const uint32_t slice = max(32u, (ns + LEAF_WARPS - 1) / LEAF_WARPS);
        const uint32_t kb = min(ns, warp * slice);
        const uint32_t end = min(ns, kb + slice);
        uint32_t nwin = 0;                                              // warp-uniform: slots this warp has claimed so far
        if (kb < end) {
            uint32_t next = kb, x = 0, tries = 0;
            uint64_t skey = 0;
            bool active = false;
            for (;;) {
                const uint32_t m = __ballot_sync(0xffffffffu, !active);
                if (m) {
                    const uint32_t idx = next + __popc(m & lane_lt);
                    next += __popc(m);
                    if (!active && idx < end) {
                        const uint32_t ki = lds16(slow_s + 2 * idx), blk = ki >> 5;
                        const uint32_t r = lds32(blk_s + 4 * blk) + __popc(lds32(mask_s + 4 * blk) & ((2u << (ki & 31u)) - 2u));
                        skey = window(r, ki - lds16(p_s + 2 * r));
                        if (CANON) skey = canon_code(skey, k);
                        x = leaf_mix(skey) * 0x2C1B3C6Du;               // decorrelate from the cell index
                        tries = 0;
                        active = true;
                    }
                }
                if (__all_sync(0xffffffffu, !active)) break;            // the warp's share is exhausted
                const uint32_t step = (x >> 6) | 1u;                    // double hashing: an odd step visits every slot
                const uint32_t h = ((x >> 22) + tries * step) & (LEAF_SLOTS - 1);
                const uint32_t slot = tbl_s + 8 * h;
                bool won = false;
                if (active) {
                    if (tries >= LEAF_SLOTS) {                          // table full: tier 2 counts this k-mer (one-k-mer record)
                        const unsigned long long si = atomicAdd(&status->n_spill, 1ull);
                        if (si < plan.spill_cap) {
                            if (RECW == 1) reinterpret_cast<unsigned long long*>(spill)[si] = skey << kshift;
                            else { ulonglong2 o; o.x = skey << kshift; o.y = 0ull; reinterpret_cast<ulonglong2*>(spill)[si] = o; }
                        } else atomicAdd(&status->n_overflow, 1ull);
                        atomicAdd(&status->n_kmers, ~0ull);            // not counted here
                        active = false;
                    } else {
                        const unsigned long long old = atoms_cas64(slot, kEmpty, skey);
                        won = old == kEmpty;
                        const bool dup = !won && (old & KEYMASK) == skey;   // !won: at k == 26 't'*26 equals kEmpty & KEYMASK
                        if (dup) {
                            if (PACKED) reds_add64(slot, 1ull << 52);
                            else reds_add32(cnt_s + 4 * h, 1u);
                        }
                        active = !(won | dup);
                        tries++;
                    }
                }
                // the claimed slots are listed in place of the warp's consumed slow-list entries (nwin < next - kb always
                // holds: every claim follows the fetch of its k-mer, and all entries below `next` have been read)
                const uint32_t wm = __ballot_sync(0xffffffffu, won);
                if (won) sts16(slow_s + 2 * (kb + nwin + __popc(wm & lane_lt)), h);
                nwin += __popc(wm);
            }
        }
        unsigned long long wbase = 0;
        if (lane == 0 && nwin && !SPEC) wbase = atomicAdd(&status->n_distinct, (unsigned long long)nwin);
        if (t == 0) s_obase[par] = ubase;
        if (RECW == 2) special_total += special;
        __syncthreads();                                                // (B) all counts final
        if (t < 2) { if (t == 0) s_nuniq[par ^ 1] = 0; else s_nslow[par ^ 1] = 0; }   // idle until the next bucket's classify phase
        if (t >= 32 && t < 32 + LEAF_BLOCKS) s_mask[par][t - 32] = 0;   // this bucket's start bits: idle until the bucket after the next
        // ---- emit the unique k-mers: coalesced 16-byte (k-mer, 1) pairs, ranks by ballot
        if (!SPEC) {
            const unsigned long long ob = s_obase[par] + woff;
            const bool fits = ob + wuniq <= (SPLIT ? capacity_u : capacity);   // uniform per warp
            if (!fits && lane == 0) status->out_overflow = 1;
            ulonglong2* const po = reinterpret_cast<ulonglong2*>(out) + ob;
            uint64_t* const pu = out_u + ob;
            uint32_t rank = 0;
            const uint32_t um = fits ? uniq : 0u;
#pragma unroll
            for (int i = 0; i < LEAF_KPT; i++) {
                if (i * LEAF_THREADS >= (int)nkeys) break;
                const bool u = (um >> i) & 1u;
                const uint32_t m = __ballot_sync(0xffffffffu, u);
                if (u) {
                    const uint32_t o = rank + __popc(m & lane_lt);
                    if (SPLIT) pu[o] = key[i];                          // split format: a bare code means count 1
                    else {
                        ulonglong2 v;
                        v.x = key[i];
                        v.y = 1ull;
                        po[o] = v;
                    }
                }
                rank += __popc(m);
            }
        }
        // ---- emit + reset the table entries this warp claimed
        if (SPEC) {
            const SpecOut so{reinterpret_cast<unsigned long long*>(out_u), capacity_u, out, capacity};
            for (uint32_t i0 = 0; i0 < nwin; i0 += 32) {               // whole warps: spectrum_bin_warp is warp-collective
                const uint32_t i = i0 + lane;
                uint64_t code = 0, cnt = 0;
                if (i < nwin) {
                    const uint32_t h = lds16(slow_s + 2 * (kb + i));
                    const unsigned long long v = lds64(tbl_s + 8 * h);
                    sts64(tbl_s + 8 * h, kEmpty);
                    unsigned long long c;
                    if (PACKED) c = v >> 52;
                    else {
                        c = lds32(cnt_s + 4 * h);
                        if (c) sts32(cnt_s + 4 * h, 0u);
                    }
                    code = v & KEYMASK;
                    cnt = 1ull + c;
                }
                spectrum_bin_warp(hist_s, so, status, code, cnt);
            }
        } else {
        wbase = __shfl_sync(0xffffffffu, wbase, 0);
        for (uint32_t i = lane; i < nwin; i += 32) {
            const uint32_t h = lds16(slow_s + 2 * (kb + i));
            const unsigned long long v = lds64(tbl_s + 8 * h);
            sts64(tbl_s + 8 * h, kEmpty);
            unsigned long long c;
            if (PACKED) c = v >> 52;
            else {
                c = lds32(cnt_s + 4 * h);
                if (c) sts32(cnt_s + 4 * h, 0u);
            }
            const uint64_t idx = wbase + i;
            if (idx < capacity) { ulonglong2 o; o.x = v & KEYMASK; o.y = 1ull + c; reinterpret_cast<ulonglong2*>(out)[idx] = o; }
            else status->out_overflow = 1;
        }
        }
        if (t == 0) kmers_total += cur.nk;
        par ^= 1;
        rb ^= 1u;
        cur = nxt;
    }
    // n_kmers counts what went through the tables; the k == 32 special key is added back by append_special_kernel
    if (RECW == 2) {
        for (int d = 16; d; d >>= 1) special_total += __shfl_xor_sync(0xffffffffu, special_total, d);
        if (lane == 0 && special_total) {
            atomicAdd(&status->special_count, special_total);
            atomicAdd(&status->n_kmers, 0ull - special_total);
        }
    }
    if (t == 0 && kmers_total) atomicAdd(&status->n_kmers, kmers_total);
    if (SPEC) {                                                         // the unique k-mers into bin 1, then the CTA's bins out
        if (lane == 0 && uniq_total) reds_add32(hist_s + 4, uniq_total);
        __syncthreads();
        spectrum_flush(hist_s, SpecOut{reinterpret_cast<unsigned long long*>(out_u), capacity_u, out, capacity});
    }
}

// ---------------------------------------------------------------------------------------------
// sharded counting, owner side: coarse partitions -> fine buckets
//
// A source GPU scatters its records over few, large coarse partitions (n_ranks * n_coarse of them: the scatter cost
// grows with the number of open regions, which must not grow with the size of the whole job).  After the exchange
// the owner splits every coarse partition into its 2^fine_shift fine buckets: one CTA per coarse partition, slot
// counters in shared memory (no global atomics), all stores of a CTA inside one small window of HBM.  The bucket of
// a record is recomputed from its first window: it is the bucket of the run's minimizer, as in partition_kernel.
template <int W, int RECW>
__global__ void __launch_bounds__(256) refine_kernel(PartitionPlan plan, int k, int n_src, uint32_t n_coarse, uint32_t coarse_cap,
                                                     const __grid_constant__ SrcTable src, unsigned long long* __restrict__ fill,
                                                     Rec<RECW>* __restrict__ recs, Rec<RECW>* __restrict__ spill, DevStatus* status) {
    extern __shared__ uint32_t refine_smem[];       // [F] records, [F] k-mers
    const uint32_t F = 1u << plan.fine_shift;
    uint32_t* s_nrec = refine_smem;
    uint32_t* s_nk = refine_smem + F;
    const int t = threadIdx.x;
    const uint32_t himask = 0xffffffffu << (32 - 2 * plan.m);
    unsigned long long overflow_kmers = 0;
    uint64_t pol_last, pol_first;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_last));
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_first));
    for (uint32_t c = blockIdx.x; c < n_coarse; c += gridDim.x) {
        for (uint32_t f = t; f < 2 * F; f += blockDim.x) refine_smem[f] = 0;
        __syncthreads();
        for (int sJ = 0; sJ < n_src; sJ++) {
            const int sI = (int)((c + (uint32_t)sJ) % (uint32_t)n_src);   // CTAs start at different sources: all links busy at all times
            const uint32_t n = min((uint32_t)ld_nc_u64(reinterpret_cast<const uint64_t*>(src.fill[sI]) + c), coarse_cap);
            const Rec<RECW>* base = reinterpret_cast<const Rec<RECW>*>(src.recs[sI]) + (uint64_t)c * coarse_cap;
            constexpr int RQ = 4;                                 // records in flight per thread
            for (uint32_t i0 = t; i0 < n; i0 += RQ * blockDim.x) {
                uint64_t hi[RQ], lo[RQ];
#pragma unroll
                for (int q = 0; q < RQ; q++) {
                    const uint32_t i = i0 + q * blockDim.x;
                    hi[q] = 0; lo[q] = 0;
                    if (i < n) {
                        if (RECW == 1) hi[q] = ld_nc_u64(reinterpret_cast<const uint64_t*>(base + i));
                        else {
                            const uint4 raw = ld_nc_u128(base + i);
                            hi[q] = ((uint64_t)raw.y << 32) | raw.x;
                            lo[q] = ((uint64_t)raw.w << 32) | raw.z;
                        }
                    }
                }
#pragma unroll
                for (int q = 0; q < RQ; q++) {
                    if (i0 + q * blockDim.x >= n) break;
                    const uint32_t L = (RECW == 1 ? (uint32_t)(hi[q] & 15u) : (uint32_t)(lo[q] & 63u)) + 1;
                    uint32_t hmin = 0xffffffffu;                  // minimizer hash of the record's first window
#pragma unroll
                    for (int j = 0; j < W; j++) {
                        const uint32_t top = (uint32_t)((hi[q] << (2 * j)) >> 32);
                        hmin = min(hmin, mmer_hash(top, himask, plan.m));
                    }
                    const uint32_t f = fine_in_coarse(bucket_position<W>(hmin, plan.even), plan.fine_shift);
                    const uint32_t slot = atomicAdd(&s_nrec[f], 1u);
                    atomicAdd(&s_nk[f], L);
                    Rec<RECW>* dst = nullptr;
                    if (slot < plan.cap) dst = recs + ((uint64_t)c * F + f) * plan.cap + slot;
                    else {                                        // region full: spill list (tier 2), else recount
                        const unsigned long long si = atomicAdd(&status->n_spill, 1ull);
                        if (si < plan.spill_cap) dst = spill + si;
                        else overflow_kmers += L;
                    }
                    if (dst) {   // same L2 policy as partition_kernel: keep a region's partially written sector resident
                        if (RECW == 1) {
                            const uint64_t pol = (slot & 3u) == 3u ? pol_first : pol_last;
                            asm volatile("st.global.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(dst), "l"(hi[q]), "l"(pol) : "memory");
                        } else {
                            const uint64_t pol = (slot & 1u) ? pol_first : pol_last;
                            asm volatile("st.global.L2::cache_hint.v2.u64 [%0], {%1, %2}, %3;" ::"l"(dst), "l"(hi[q]), "l"(lo[q]), "l"(pol) : "memory");
                        }
                    }
                }
            }
        }
        __syncthreads();
        for (uint32_t f = t; f < F; f += blockDim.x)
            fill[(uint64_t)c * F + f] = ((unsigned long long)s_nk[f] << 32) | s_nrec[f];
        __syncthreads();
    }
    if (overflow_kmers) atomicAdd(&status->n_overflow, overflow_kmers);
}

// The same split for 8-byte records (k <= 26), with write combining.  Scattered 8-byte stores are what limits the direct
// version (~70 G stores/s: every one is a read-modify-write of a 32-byte sector in L2).  Here the CTA takes its coarse partition
// in rounds of 1024 records, counting-sorts a round by fine bucket in shared memory, and thread f appends bucket f's records as
// whole, aligned 32-byte sectors (one 256-bit store for four records); what does not fill a sector waits in a 3-record carry
// buffer per bucket for the next round.
constexpr int RF_ROUND = 1024;          // records per round (4 per thread)
template <int W>
__global__ void __launch_bounds__(256) refine_staged_kernel(PartitionPlan plan, int k, int n_src, uint32_t n_coarse, uint32_t coarse_cap,
                                                            const __grid_constant__ SrcTable src, unsigned long long* __restrict__ fill,
                                                            Rec<1>* __restrict__ recs, Rec<1>* __restrict__ spill, DevStatus* status) {
    constexpr int F = 256;                                   // fine buckets per coarse partition == threads per CTA
    __shared__ uint32_t s_hist[F], s_start[F], s_gk[F], s_wtot[8], s_n[KMER_MAX_SRC];
    __shared__ __align__(16) unsigned long long s_sorted[RF_ROUND];
    __shared__ unsigned long long s_carry[3][F];             // bucket t's pending records: s_carry[0..n_carry)[t]
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const uint32_t himask = 0xffffffffu << (32 - 2 * plan.m);
    const uint32_t cap = plan.cap;                           // a multiple of 4 (make_partition_plan): regions are whole sectors
    unsigned long long overflow_kmers = 0;
    for (uint32_t c = blockIdx.x; c < n_coarse; c += gridDim.x) {
        uint32_t gpos = 0, n_carry = 0, n_total = 0;         // bucket t: records written to its region (a multiple of 4) / pending / all
        unsigned long long* const dst = reinterpret_cast<unsigned long long*>(recs + ((uint64_t)c * F + t) * plan.cap);
        auto put_spill = [&](unsigned long long r) {         // region full: spill list (tier 2), else recount
            const unsigned long long si = atomicAdd(&status->n_spill, 1ull);
            if (si < plan.spill_cap) reinterpret_cast<unsigned long long*>(spill)[si] = r;
            else overflow_kmers += (r & 15u) + 1;
        };
        s_gk[t] = 0;
        // the sources' segment sizes, all at once (a source may be another GPU's memory: one round trip, not n_src)
        // position j of the order is source (c + j) % n_src: CTAs start at different sources, so that all GPUs' links are busy at
        // all times (in the same order everywhere, every owner would read from the same GPU at the same moment)
        if (t < n_src) s_n[t] = min((uint32_t)ld_nc_u64(reinterpret_cast<const uint64_t*>(src.fill[(c + t) % n_src]) + c), coarse_cap);
        __syncthreads();
        // rounds of RF_ROUND records over all sources; the loads of the next round are issued before this one is processed
        auto seek = [&](int& sI, uint32_t& r0) {             // first (source, round) at or after (sI, r0) that holds records
            while (sI < n_src && r0 >= s_n[sI]) { sI++; r0 = 0; }
        };
        auto fetch = [&](int sI, uint32_t r0, uint64_t (&rec)[4]) {
            const uint64_t* base = reinterpret_cast<const uint64_t*>(src.recs[(c + (uint32_t)sI) % (uint32_t)n_src]) + (uint64_t)c * coarse_cap;
            const uint32_t n = s_n[sI];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint32_t i = r0 + q * 256 + t;
                rec[q] = i < n ? ld_nc_u64(base + i) : 0ull;
            }
        };
        int sI = 0;
        uint32_t r0 = 0;
        uint64_t rec[4], nxt[4];
        seek(sI, r0);
        if (sI < n_src) fetch(sI, r0, rec);
        while (sI < n_src) {
            const uint32_t n = s_n[sI], r0c = r0;
            int sN = sI;
            uint32_t rN = r0 + RF_ROUND;
            seek(sN, rN);
            if (sN < n_src) fetch(sN, rN, nxt);
            {
                s_hist[t] = 0;
                __syncthreads();                              // histogram zeroed; previous round fully consumed
                uint32_t fr[4];                               // fine bucket << 16 | rank within the round
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    fr[q] = 0xffffffffu;
                    if (r0c + q * 256 + t < n) {
                        uint32_t hmin = 0xffffffffu;          // minimizer hash of the record's first window
#pragma unroll
                        for (int j = 0; j < W; j++) {
                            const uint32_t top = (uint32_t)((rec[q] << (2 * j)) >> 32);
                            hmin = min(hmin, mmer_hash(top, himask, plan.m));
                        }
                        const uint32_t f = fine_in_coarse(bucket_position<W>(hmin, plan.even), plan.fine_shift);
                        fr[q] = (f << 16) | atomicAdd(&s_hist[f], 1u);
                        atomicAdd(&s_gk[f], (uint32_t)(rec[q] & 15u) + 1);
                    }
                }
                __syncthreads();
                // exclusive scan of the histogram: one bucket per thread
                const uint32_t cnt = s_hist[t];
                uint32_t incl = cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += v;
                }
                if (lane == 31) s_wtot[warp] = incl;
                __syncthreads();
                uint32_t st0 = incl - cnt;
#pragma unroll
                for (int q = 0; q < 8; q++)
                    if (q < warp) st0 += s_wtot[q];
                s_start[t] = st0;
                __syncthreads();
#pragma unroll
                for (int q = 0; q < 4; q++)
                    if (fr[q] != 0xffffffffu) s_sorted[s_start[fr[q] >> 16] + (fr[q] & 0xffffu)] = rec[q];
                __syncthreads();
                // thread t: bucket t's pending records followed by this round's, as whole sectors; the rest is carried on
                if (cnt) {
                    n_total += cnt;
                    const uint32_t total = n_carry + cnt;
                    auto item = [&](uint32_t j) { return j < n_carry ? s_carry[j][t] : s_sorted[st0 + (j - n_carry)]; };
                    uint32_t j = 0;
                    for (; j + 4 <= total; j += 4) {
                        const unsigned long long r0v = item(j), r1v = item(j + 1), r2v = item(j + 2), r3v = item(j + 3);
                        if (gpos + 4 <= cap) {
                            asm volatile("st.global.v4.u64 [%0], {%1, %2, %3, %4};" ::"l"(dst + gpos), "l"(r0v), "l"(r1v), "l"(r2v), "l"(r3v) : "memory");
                            gpos += 4;
                        } else { put_spill(r0v); put_spill(r1v); put_spill(r2v); put_spill(r3v); }
                    }
                    const uint32_t left = total - j;          // 0..3
                    unsigned long long keep[3];
#pragma unroll
                    for (uint32_t q = 0; q < 3; q++) keep[q] = q < left ? item(j + q) : 0ull;
#pragma unroll
                    for (uint32_t q = 0; q < 3; q++)
                        if (q < left) s_carry[q][t] = keep[q];
                    n_carry = left;
                }
            }
            sI = sN; r0 = rN;
#pragma unroll
            for (int q = 0; q < 4; q++) rec[q] = nxt[q];
        }
        // the last, partial sector of every bucket (the region fills up completely before anything is spilled, so
        // min(records, cap) of them are in the region and records > cap marks the overflow, as partition_kernel leaves it)
        for (uint32_t q = 0; q < n_carry; q++) {
            if (gpos < cap) dst[gpos + q] = s_carry[q][t];
            else put_spill(s_carry[q][t]);
        }
        __syncthreads();
        fill[(uint64_t)c * F + t] = ((unsigned long long)s_gk[t] << 32) | (uint64_t)n_total;
        __syncthreads();
    }
    if (overflow_kmers) atomicAdd(&status->n_overflow, overflow_kmers);
}

// tier 2: every k-mer of the failed buckets (their in-region records) and of the spill list goes into
// a global open-addressing table (count_hash.cu layout); hash_compact then appends it to the result.
// Failed buckets and spilled records hold k-mers of the same buckets only, so nothing here can also
// have been emitted by bucket_count_kernel.
__device__ __forceinline__ void global_table_add(kmer_count_pair* slots, uint64_t mask, uint64_t code, unsigned long long c) {
    uint64_t h = mix64(code) & mask;
    for (;;) {
        unsigned long long prev = atomicCAS((unsigned long long*)&slots[h].code, kEmpty, code);
        if (prev == kEmpty || prev == code) { atomicAdd((unsigned long long*)&slots[h].count, c); return; }
        h = (h + 1) & mask;
    }
}

template <int RECW, bool CANON>
__device__ __forceinline__ void tier2_add_record(const Rec<RECW>* p, int kshift, kmer_count_pair* slots, uint64_t mask,
                                                 DevStatus* status, bool active) {
    uint64_t hi = 0, lo = 0;
    int L = 0;
    if (active) {
        if (RECW == 1) { hi = reinterpret_cast<const uint64_t*>(p)[0]; L = (int)(hi & 15u) + 1; }
        else { hi = reinterpret_cast<const uint64_t*>(p)[0]; lo = reinterpret_cast<const uint64_t*>(p)[1]; L = (int)(lo & 63u) + 1; }
    }
    const int lane = threadIdx.x & 31;
    int maxL = L;
    for (int d = 16; d; d >>= 1) maxL = max(maxL, __shfl_xor_sync(0xffffffffu, maxL, d));
    for (int o = 0; o < maxL; o++) {
        bool v = o < L;
        uint64_t win = (RECW == 1 || o == 0) ? (hi << (2 * o)) : ((hi << (2 * o)) | (lo >> (64 - 2 * o)));
        uint64_t key = win >> kshift;
        if (CANON) key = canon_code(key, (64 - kshift) >> 1);   // the leaf's one-k-mer spill records are canonical already
        uint32_t vm = __ballot_sync(0xffffffffu, v);
        uint32_t same = __match_any_sync(0xffffffffu, key) & vm;     // repetitive input: aggregate equal keys
        if (v && lane == __ffs(same) - 1) {
            unsigned long long c = __popc(same);
            if (key == kEmpty) atomicAdd(&status->special_count, c);
            else global_table_add(slots, mask, key, c);
        }
    }
}

// one thread: does tier 2 have to run, and does what it must count fit its table?
__global__ void tier2_decide_kernel(PartitionPlan plan, uint64_t n_slots, DevStatus* status) {
    const unsigned long long spilled = min(status->n_spill, (unsigned long long)plan.spill_cap);
    unsigned long long mode = 0, slots = 0;
    if (status->n_overflow) mode = 2;                                   // the spill list overflowed: the batch is recounted
    else if (status->n_failed || status->n_spill) {
        const unsigned long long need = (status->failed_kmers + spilled * 16ull) * 2ull;   // load factor <= 1/2
        mode = 1;
        slots = 1024;
        while (slots < need && slots < n_slots) slots <<= 1;
        if (slots < need) { mode = 2; atomicAdd(&status->n_overflow, 1ull); }
    }
    status->t2_mode = mode;
    status->t2_slots = slots;
}

__global__ void __launch_bounds__(256) tier2_clear_kernel(uint4* __restrict__ slots, const DevStatus* status) {
    if (status->t2_mode != 1ull) return;
    const uint64_t n_slots = status->t2_slots;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_slots; i += stride) slots[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
}

template <int RECW, bool CANON = false>
__global__ void __launch_bounds__(256) tier2_insert_kernel(PartitionPlan plan, int k, const unsigned long long* __restrict__ fill,
                                                           const Rec<RECW>* __restrict__ recs, const uint32_t* __restrict__ failed_ids,
                                                           const Rec<RECW>* __restrict__ spill, kmer_count_pair* __restrict__ slots,
                                                           DevStatus* status) {
    if (status->t2_mode != 1ull) return;
    const uint64_t mask = status->t2_slots - 1;
    const int kshift = 64 - 2 * k;
    const uint32_t n_failed = (uint32_t)status->n_failed;
    for (uint32_t fi = blockIdx.x; fi < n_failed; fi += gridDim.x) {
        const uint32_t b = failed_ids[fi];
        const uint32_t nrec = min((uint32_t)fill[b] & 0x7fffffffu, plan.cap);   // bit 31: poison (scatter.cuh)
        const Rec<RECW>* base = recs + (uint64_t)b * plan.cap;
        for (uint32_t r0 = 0; r0 < nrec; r0 += blockDim.x) {
            uint32_t r = r0 + threadIdx.x;
            tier2_add_record<RECW, CANON>(base + min(r, nrec - 1), kshift, slots, mask, status, r < nrec);
        }
    }
    const uint64_t n_spill = min((uint64_t)status->n_spill, (uint64_t)plan.spill_cap);
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t r0 = (uint64_t)blockIdx.x * blockDim.x; r0 < n_spill; r0 += stride) {
        uint64_t r = r0 + threadIdx.x;
        tier2_add_record<RECW, CANON>(spill + min(r, n_spill - 1), kshift, slots, mask, status, r < n_spill);
    }
}

// appends the k == 32 all-ones key, whose occurrences were kept out of the tables
__global__ void append_special_kernel(kmer_count_pair* out, uint64_t capacity, DevStatus* status) {
    unsigned long long sc = status->special_count;
    if (!sc) return;
    unsigned long long idx = atomicAdd(&status->n_distinct, 1ull);
    if (idx < capacity) { out[idx].code = kEmpty; out[idx].count = sc; }
    else status->out_overflow = 1;
    atomicAdd(&status->n_kmers, sc);
}

}  // namespace kmer
#include "scatter.cuh"
namespace kmer {

// ---------------------------------------------------------------------------------------------
// host side

static double poisson_tail(double lam, int c) {          // P(X > c), X ~ Poisson(lam)
    double term = exp(-lam), cdf = term;
    for (int i = 1; i <= c; i++) { term *= lam / i; cdf += term; }
    return cdf >= 1.0 ? 0.0 : 1.0 - cdf;
}
// staging slots per destination: a sector's leftover (sect - 1) plus the arrivals of one round, so that a round needs
// a second flush (a destination's slots taken) with probability < budget
static uint32_t stage_slots(double lam, uint32_t sect, double dests, double budget, uint32_t max_slots) {
    uint32_t c;
    if (lam > 30.0) c = (uint32_t)(lam + 6.0 * sqrt(lam)) + sect;      // normal tail (few, large destinations: small jobs)
    else {
        c = sect;
        while (c < max_slots && dests * poisson_tail(lam, (int)(c - (sect - 1))) > budget) c++;
    }
    return c < max_slots ? c : max_slots;
}
static size_t stage_fixed_bytes(uint32_t dests) { return (((size_t)dests * 12 + 8 + 15) & ~(size_t)15) + 16; }   // Stage: cnt, gpos, rdy lists
static size_t stage_bytes(uint32_t dests, uint32_t caps, int recw) { return stage_fixed_bytes(dests) + (size_t)dests * caps * (recw == 1 ? 8 : 16); }
static size_t scatter_static_smem() { return sizeof(ScanSmem) + (NT / 32) * SCAT_RUNCAP * 6 + (TILE / 32 + 2) * 4 + 64; }

bool make_scatter_plan(const DeviceInfo& di, uint64_t n_bases, uint64_t n_kmers, PartitionPlan& p, ScatterPlan& sp) {
    uint32_t fine_shift = 10;                              // F = 1024 fine buckets per coarse partition: one per refine2 thread
#ifdef KMER_TUNE
    if (const char* e = getenv("KMER_FINE_SHIFT")) fine_shift = (uint32_t)atoi(e);
#endif
    while (fine_shift > 0 && (1u << fine_shift) > p.n_buckets) fine_shift--;
    const uint64_t D = ((uint64_t)p.n_buckets + (1u << fine_shift) - 1) >> fine_shift;
    if (D > (uint64_t)SCAT_DPT * NT || fine_shift > 10) return false;
    const double rpk = 2.1 / (p.w + 1) + (p.rmax < p.w ? 1.0 / p.rmax : 0.0);   // records per k-mer (make_partition_plan)
    const uint32_t sect = p.recw == 1 ? 4 : 2;
    const uint64_t n_tiles = (n_bases + TILE - 1) / TILE;
    // pass 1: as many CTAs per SM as the staging area allows (at most SCAT_MINB)
    uint32_t caps = 0, per_sm = SCAT_MINB;
    for (; per_sm >= 1; per_sm--) {
        const size_t budget = (size_t)227 * 1024 / per_sm - 1024 - scatter_static_smem();
        const uint32_t max_slots = (uint32_t)std::min<size_t>(4096, (budget - stage_fixed_bytes((uint32_t)D)) / (D * (p.recw == 1 ? 8 : 16)));
        if (max_slots < sect + 2) continue;
        caps = stage_slots(TILE * rpk / (double)D, sect, (double)D, 0.02, max_slots);
        if (caps < max_slots || per_sm == 1) break;       // the slots wanted fit (or nothing smaller is left to try)
    }
    if (per_sm < 1 || caps < sect) return false;
#ifdef KMER_TUNE
    if (const char* e = getenv("KMER_SCAT_CAPS")) caps = (uint32_t)atoi(e);
    if (const char* e = getenv("KMER_SCAT_PER_SM")) per_sm = (uint32_t)atoi(e);
#endif
    uint64_t grid = (uint64_t)di.sm_count * per_sm;
    if (grid > n_tiles) grid = n_tiles ? n_tiles : 1;
    const double mean = (double)n_kmers * rpk / ((double)grid * (double)D);
    sp.n_coarse = (uint32_t)D;
    sp.n_src = (uint32_t)grid;
    sp.seg_cap = ((uint32_t)(1.1 * mean + 6.0 * sqrt(mean) + 32.0) + 3u) & ~3u;
    sp.caps = caps;
    const uint32_t F = 1u << fine_shift;
    const size_t budget2 = (size_t)227 * 1024 - 1024 - (((size_t)F * 4 + 15) & ~(size_t)15) - stage_fixed_bytes(F);
    const uint32_t max2 = (uint32_t)std::min<size_t>(4096, budget2 / ((size_t)F * (p.recw == 1 ? 8 : 16)));
    sp.caps2 = stage_slots((double)RF2_THREADS * RF2_RQ / (double)F, sect, (double)F, 0.02, max2);
    p.n_buckets = (uint32_t)(D << fine_shift);
    p.hash_buckets = p.n_buckets;
    p.fine_shift = (int)fine_shift;
    const uint64_t sc = (uint64_t)p.n_buckets * p.cap / 8;
    p.spill_cap = sc < 4096 ? 4096 : sc;
    return true;
}

size_t scatter_seg_bytes(const PartitionPlan& p, const ScatterPlan& sp) {
    return (size_t)sp.n_src * sp.n_coarse * sp.seg_cap * (p.recw == 1 ? 8 : 16);
}
size_t scatter_segfill_bytes(const ScatterPlan& sp) { return (size_t)sp.n_src * sp.n_coarse * 4; }

template <int W, int RECW>
static void launch_scatter_refine_t(const DeviceInfo& di, const ScanArgs& a, const PartitionPlan& p, const ScatterPlan& sp, uint32_t* d_segfill,
                                    void* d_seg, unsigned long long* d_fill, void* d_recs, void* d_spill, cudaStream_t st,
                                    void (*mark)(void*, const char*), void* mark_arg) {
    static size_t conf1[64] = {}, conf2[64] = {};          // per device: dynamic shared memory opted in so far
    int dev = 0;
    cudaGetDevice(&dev);
    const size_t smem1 = stage_bytes(sp.n_coarse, sp.caps, RECW);
    const size_t smem2 = ((((size_t)4 << p.fine_shift) + 15) & ~(size_t)15) + stage_bytes(1u << p.fine_shift, sp.caps2, RECW);
    if (dev >= 0 && dev < 64 && conf1[dev] < smem1) {
        cudaFuncSetAttribute(scatter_kernel<W, RECW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1);
        cudaFuncSetAttribute(scatter_kernel<W, RECW>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        conf1[dev] = smem1;
    }
    if (dev >= 0 && dev < 64 && conf2[dev] < smem2) {
        cudaFuncSetAttribute(refine2_kernel<W, RECW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
        cudaFuncSetAttribute(refine2_kernel<W, RECW>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        conf2[dev] = smem2;
    }
    cudaMemsetAsync(d_fill, 0, (size_t)p.n_buckets * sizeof(unsigned long long), st);
    scatter_kernel<W, RECW><<<sp.n_src, NT, smem1, st>>>(a, p, sp, d_segfill, (Rec<RECW>*)d_seg, d_fill, (Rec<RECW>*)d_spill);
    if (mark) mark(mark_arg, "scatter");
    unsigned grid2 = (unsigned)std::min<uint64_t>(sp.n_coarse, (uint64_t)di.sm_count);
    refine2_kernel<W, RECW><<<grid2, RF2_THREADS, smem2, st>>>(p, sp, d_segfill, (const Rec<RECW>*)d_seg, d_fill, (Rec<RECW>*)d_recs,
                                                                (Rec<RECW>*)d_spill, a.status);
    if (mark) mark(mark_arg, "refine");
}

void launch_scatter_refine(const DeviceInfo& di, const ScanArgs& a, const PartitionPlan& p, const ScatterPlan& sp, uint32_t* d_segfill,
                           void* d_seg, unsigned long long* d_fill, void* d_recs, void* d_spill, cudaStream_t st,
                           void (*mark)(void*, const char*), void* mark_arg) {
#define KMER_SR(W_, R_) launch_scatter_refine_t<W_, R_>(di, a, p, sp, d_segfill, d_seg, d_fill, d_recs, d_spill, st, mark, mark_arg)
    if (p.recw == 1) {
        if (p.w == 4) KMER_SR(4, 1);
        else if (p.w == 6) KMER_SR(6, 1);
        else if (p.w == 9) KMER_SR(9, 1);
        else KMER_SR(8, 1);
    } else {
        if (p.w == 8) KMER_SR(8, 2);
        else if (p.w == 12) KMER_SR(12, 2);
        else KMER_SR(16, 2);
    }
#undef KMER_SR
}


static int g_forced_window = 0;
void partition_force_window(int w) { g_forced_window = w; }

// m-mer length for window w: k - w + 1, capped at 16 bases.  Canonical counting (partition_kernel<.., true>) centres the w m-mers
// in the k-mer, which needs k - w + 1 - m even, and has only about 4^m / 2 distinct (canonical) m-mers.
static int plan_m(int k, int w, bool canon) {
    int m = k - w + 1 > 16 ? 16 : k - w + 1;
    if (canon && ((k - w + 1 - m) & 1)) m--;
    return m;
}
static bool mmers_fine_enough(int m, bool canon, uint64_t nb) { return ldexp(1.0, 2 * m - (canon ? 1 : 0)) >= 30.0 * (double)nb; }

PartitionPlan make_partition_plan(uint64_t n_kmers, int k, bool canon) {
    PartitionPlan p{};
    // minimizer window: w windows share a record while their minimizer (an m-mer, m = k - w + 1, capped at 16 bases) stays the same
    const uint32_t target = TARGET_KMERS_PER_BUCKET;
    uint64_t nb = (n_kmers + target - 1) / target;
    if (nb < 1) nb = 1;
    if (nb > 0x7fffffffull) nb = 0x7fffffffull;
    p.recw = k <= 26 ? 1 : 2;
    // The widest window (fewest records: about 2/(w+1) per k-mer) whose m-mers are still fine-grained enough for the buckets: a
    // bucket covers a range of the minimizer order of equal expected load (minimizer_rank), but it cannot split an m-mer, and one
    // frequent m-mer is the minimizer of up to w windows per occurrence.  4^m >= 30 * buckets keeps that below ~1/4 of a bucket
    // (simulated: 0.3 % of the k-mers in buckets above the on-chip limit at 41 m-mers per bucket, ~1 % at 30; they go to tier 2).
    // n_kmers is the size of the WHOLE job.  9 windows need k = 21 or 22: a 13-base m-mer and 9 windows in an 8-byte record.
    {
        static const int ws1[] = {9, 8, 6, 4}, ws2[] = {16, 16, 12, 8};
        const int* ws = p.recw == 1 ? ws1 : ws2;
        p.w = ws[3];
        p.even = 1;                                        // nothing fits: the narrowest window, m-mers spread by a second hash
        for (int i = 0; i < 4; i++) {
            const int m = plan_m(k, ws[i], canon);
            if (ws[i] == 9 && k > 22) continue;            // 9 windows do not fit an 8-byte record (30 bases) beyond k = 22
            if (mmers_fine_enough(m, canon, nb)) { p.w = ws[i]; p.even = 0; break; }
        }
    }
    if (g_forced_window) {                                 // tests only (kmer_cuda_test_force_window): must suit the record width and k
        const int w = g_forced_window;
        const bool ok = p.recw == 1 ? (w == 4 || w == 6 || w == 8 || w == 9) : (w == 8 || w == 12 || w == 16);
        if (ok && k - w + 1 >= 2) {
            p.w = w;
            p.even = mmers_fine_enough(plan_m(k, w, canon), canon, nb) ? 0 : 1;
        }
    }
    p.m = plan_m(k, p.w, canon);
    p.rmax = p.recw == 1 ? (30 - k + 1 > 16 ? 16 : 30 - k + 1) : 16;
    p.n_buckets = (uint32_t)nb;
    p.hash_buckets = p.n_buckets;
    p.fine_shift = 0;
    {   // records per bucket: about 2/(w+1) records per k-mer (runs end where the minimizer changes, and at tile borders)
        const double rpk = 2.1 / (p.w + 1) + (p.rmax < p.w ? 1.0 / p.rmax : 0.0);
        const double mean = target * rpk;
        p.cap = ((uint32_t)(1.25 * mean + 5.0 * sqrt(3.0 * mean) + 16.0) + 3u) & ~3u;   // whole 32-byte sectors of 8-byte records
    }
    uint64_t sc = (uint64_t)p.n_buckets * p.cap / 8;          // spill list: 1/8 of the bucket regions
    p.spill_cap = sc < 4096 ? 4096 : sc;
    return p;
}

size_t partition_record_bytes(const PartitionPlan& p) { return (size_t)p.n_buckets * p.cap * (p.recw == 1 ? 8 : 16); }
size_t partition_spill_bytes(const PartitionPlan& p) { return (size_t)p.spill_cap * (p.recw == 1 ? 8 : 16); }

void launch_partition(const DeviceInfo& di, const ScanArgs& a, const PartitionPlan& p, unsigned long long* d_fill,
                      void* d_recs, void* d_spill, cudaStream_t st, bool clear_fill, bool canon) {
    if (clear_fill) cudaMemsetAsync(d_fill, 0, (size_t)p.n_buckets * sizeof(unsigned long long), st);
    uint64_t n_tiles = a.tile_end ? a.tile_end - a.tile_begin : (a.n_bases + TILE - 1) / TILE;
    uint64_t grid = (uint64_t)di.sm_count * PART_MINB;
    if (grid > n_tiles) grid = n_tiles;
    if (!n_tiles) return;
#define KMER_PART(W_, R_) partition_kernel<W_, R_, C_><<<(unsigned)grid, NT, 0, st>>>(a, p, d_fill, (Rec<R_>*)d_recs, (Rec<R_>*)d_spill)
#define KMER_PART_ALL                                                                 \
    if (p.w == 4) KMER_PART(4, 1);                                                    \
    else if (p.w == 6) KMER_PART(6, 1);                                               \
    else if (p.w == 9) KMER_PART(9, 1);                                               \
    else if (p.w == 12) KMER_PART(12, 2);                                             \
    else if (p.w == 8 && p.recw == 1) KMER_PART(8, 1);                                \
    else if (p.w == 8) KMER_PART(8, 2);                                               \
    else KMER_PART(16, 2)
    if (canon) {
        constexpr bool C_ = true;
        KMER_PART_ALL;
    } else {
        constexpr bool C_ = false;
        KMER_PART_ALL;
    }
#undef KMER_PART_ALL
#undef KMER_PART
}

// p.n_buckets = buckets counted HERE (all of them on one GPU, the owned range when sharded)
size_t leaf_smem_bytes(const PartitionPlan& p) {
    const size_t recb = p.recw == 1 ? 8 : 16;
    size_t fixed = (size_t)LEAF_SLOTS * 8 + (p.recw == 1 ? 0 : (size_t)LEAF_SLOTS * 4) + 2 * (size_t)LEAF_CELLS / 8 + (size_t)LEAF_KEYS * 2 +
                   ((((size_t)p.cap + 2) * 2 + 15) & ~(size_t)15);
    size_t staged = ((size_t)p.cap + 2) * recb;                           // padded to 16 bytes
    return fixed + 2 * ((staged + 15) & ~(size_t)15);                     // two record buffers
}

// once per process and device: opt in to the leaf's dynamic shared memory (the spectrum format adds its bins)
static void leaf_configure(size_t smem) {
    static size_t configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || configured[dev] >= smem) return;
#define KMER_LEAF_CONF(RW, ...)                                                                                         \
    cudaFuncSetAttribute(bucket_count_kernel<RW, __VA_ARGS__>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem + SPEC_SBINS * 4); \
    cudaFuncSetAttribute(bucket_count_kernel<RW, __VA_ARGS__>, cudaFuncAttributePreferredSharedMemoryCarveout, 100)
    KMER_LEAF_CONF(1, false); KMER_LEAF_CONF(1, true); KMER_LEAF_CONF(2, false); KMER_LEAF_CONF(2, true);
    KMER_LEAF_CONF(1, false, true); KMER_LEAF_CONF(2, false, true);
    KMER_LEAF_CONF(1, false, false, true); KMER_LEAF_CONF(1, true, false, true); KMER_LEAF_CONF(2, false, false, true);
    KMER_LEAF_CONF(2, true, false, true); KMER_LEAF_CONF(1, false, true, true); KMER_LEAF_CONF(2, false, true, true);
#undef KMER_LEAF_CONF
    configured[dev] = smem;
}

void launch_bucket_count(const DeviceInfo& di, const PartitionPlan& p, int k, const unsigned long long* d_fill,
                         const void* d_recs, void* d_spill, uint32_t* d_failed_ids, kmer_count_pair* d_pairs, uint64_t capacity,
                         uint64_t* d_uniq, uint64_t uniq_capacity, DevStatus* d_status, cudaStream_t st, uint32_t bucket_begin,
                         uint32_t bucket_end, const SpecOut* spec, bool canon) {
    if (bucket_end == 0 || bucket_end > p.n_buckets) bucket_end = p.n_buckets;
    if (bucket_begin >= bucket_end) return;
    const size_t leaf_smem = leaf_smem_bytes(p) + (spec ? SPEC_SBINS * 4 : 0);
    int per_sm = (int)((size_t)227 * 1024 / (leaf_smem + 1024));
    if (per_sm > LEAF_MINB) per_sm = LEAF_MINB;
    if (per_sm < 1) per_sm = 1;
    uint64_t lgrid = (uint64_t)di.sm_count * per_sm;
    if (lgrid > bucket_end - bucket_begin) lgrid = bucket_end - bucket_begin;
    leaf_configure(leaf_smem_bytes(p));
#define KMER_LEAF_SPEC(RW, CN)                                                                                                    \
    bucket_count_kernel<RW, false, true, CN><<<(unsigned)lgrid, LEAF_THREADS, leaf_smem, st>>>(                                    \
        p, k, d_fill, (const Rec<RW>*)d_recs, spec->tail, spec->tail_cap, reinterpret_cast<uint64_t*>(spec->hist), spec->hist_len, \
        d_failed_ids, (Rec<RW>*)d_spill, d_status, bucket_begin, bucket_end)
#define KMER_LEAF_GO(RW, SP, CN)                                                                                                        \
    bucket_count_kernel<RW, SP, false, CN><<<(unsigned)lgrid, LEAF_THREADS, leaf_smem, st>>>(p, k, d_fill, (const Rec<RW>*)d_recs, d_pairs, capacity, \
                                                                                  d_uniq, uniq_capacity, d_failed_ids, (Rec<RW>*)d_spill, d_status, bucket_begin, bucket_end)
#define KMER_LEAF_ALL(CN)                                                                                    \
    if (spec) {                                                                                              \
        if (p.recw == 1) KMER_LEAF_SPEC(1, CN);                                                              \
        else KMER_LEAF_SPEC(2, CN);                                                                          \
    } else if (p.recw == 1) { if (d_uniq) KMER_LEAF_GO(1, true, CN); else KMER_LEAF_GO(1, false, CN); }      \
    else { if (d_uniq) KMER_LEAF_GO(2, true, CN); else KMER_LEAF_GO(2, false, CN); }
    if (canon) { KMER_LEAF_ALL(true) }
    else { KMER_LEAF_ALL(false) }
#undef KMER_LEAF_ALL
#undef KMER_LEAF_GO
#undef KMER_LEAF_SPEC
}

void launch_count_partition(const DeviceInfo& di, const ScanArgs& a, const PartitionPlan& p, unsigned long long* d_fill,
                            void* d_recs, void* d_spill, uint32_t* d_failed_ids, kmer_count_pair* d_pairs, uint64_t capacity,
                            uint64_t* d_uniq, uint64_t uniq_capacity, cudaStream_t st, void (*mark)(void*, const char*), void* mark_arg,
                            const SpecOut* spec, bool canon) {
    launch_partition(di, a, p, d_fill, d_recs, d_spill, st, true, canon);
    if (mark) mark(mark_arg, "minimizer_partition");
    launch_bucket_count(di, p, a.k, d_fill, d_recs, d_spill, d_failed_ids, d_pairs, capacity, d_uniq, uniq_capacity, a.status, st, 0, 0,
                        spec, canon);
    if (mark) mark(mark_arg, "bucket_count");
}

uint64_t tier2_table_slots(uint64_t n_kmers) {
    uint64_t want = n_kmers / 4, p = 1ull << 16;                      // room for 1/8 of the k-mers at load factor 1/2
    while (p < want) p <<= 1;
    return p;
}

void launch_partition_tier2(const DeviceInfo& di, const PartitionPlan& p, int k, const unsigned long long* d_fill,
                            const void* d_recs, const void* d_spill, const uint32_t* d_failed_ids, kmer_count_pair* d_slots,
                            uint64_t n_slots, kmer_count_pair* d_pairs, uint64_t capacity, DevStatus* d_status, cudaStream_t st,
                            void (*mark)(void*, const char*), void* mark_arg, const SpecOut* spec, bool canon) {
    const unsigned grid = (unsigned)di.sm_count * 8;
    tier2_decide_kernel<<<1, 1, 0, st>>>(p, n_slots, d_status);
    tier2_clear_kernel<<<grid, 256, 0, st>>>((uint4*)d_slots, d_status);
#define KMER_T2(R_, C_) tier2_insert_kernel<R_, C_><<<grid, 256, 0, st>>>(p, k, d_fill, (const Rec<R_>*)d_recs, d_failed_ids, \
                                                                       (const Rec<R_>*)d_spill, d_slots, d_status)
    if (p.recw == 1) { if (canon) KMER_T2(1, true); else KMER_T2(1, false); }
    else { if (canon) KMER_T2(2, true); else KMER_T2(2, false); }
#undef KMER_T2
    if (mark) mark(mark_arg, "tier2_insert");
    if (spec) launch_hash_spectrum(di, d_slots, n_slots, k, *spec, d_status, st, 1);   // + the k == 32 special key
    else launch_hash_compact(di, d_slots, n_slots, k, d_pairs, capacity, d_status, st, 1);
    if (mark) mark(mark_arg, spec ? "tier2_spectrum" : "tier2_compact");
}

void launch_refine(const DeviceInfo& di, const PartitionPlan& p, int k, int n_src, uint32_t n_coarse, uint32_t coarse_cap,
                   const SrcTable& src, unsigned long long* d_fill, void* d_recs, void* d_spill, DevStatus* d_status, cudaStream_t st) {
    if (!n_coarse) return;
    unsigned grid = (unsigned)di.sm_count * 8;
    if (grid > n_coarse) grid = n_coarse;
    const size_t smem = (size_t)(2u << p.fine_shift) * sizeof(uint32_t);
    if (p.recw == 1 && p.fine_shift == 8) {   // write-combining version (8-byte records)
#define KMER_RS(W_) refine_staged_kernel<W_><<<grid, 256, 0, st>>>(p, k, n_src, n_coarse, coarse_cap, src, d_fill, (Rec<1>*)d_recs, (Rec<1>*)d_spill, d_status)
        if (p.w == 4) KMER_RS(4);
        else if (p.w == 6) KMER_RS(6);
        else if (p.w == 9) KMER_RS(9);
        else KMER_RS(8);
#undef KMER_RS
        return;
    }
#define KMER_RF(W_, R_) refine_kernel<W_, R_><<<grid, 256, smem, st>>>(p, k, n_src, n_coarse, coarse_cap, src, d_fill, (Rec<R_>*)d_recs, (Rec<R_>*)d_spill, d_status)
    if (p.w == 6) KMER_RF(6, 1);
    else if (p.w == 12) KMER_RF(12, 2);
    else if (p.w == 4) KMER_RF(4, 1);
    else if (p.w == 9) KMER_RF(9, 1);
    else if (p.w == 8 && p.recw == 1) KMER_RF(8, 1);
    else if (p.w == 8) KMER_RF(8, 2);
    else KMER_RF(16, 2);
#undef KMER_RF
}

void launch_append_special(kmer_count_pair* d_pairs, uint64_t capacity, DevStatus* d_status, cudaStream_t st) {
    append_special_kernel<<<1, 1, 0, st>>>(d_pairs, capacity, d_status);
}

}  // namespace kmer
