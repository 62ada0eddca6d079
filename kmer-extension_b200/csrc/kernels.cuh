// kernels.cuh -- launch wrappers implemented across the .cu files of libkmer_cuda.so
#pragma once
#include "common.cuh"
#include "scan.cuh"
#include "../../include/kmer_cuda.h"

namespace kmer {

// number of CTAs the tile-scanning kernels are launched with (filled at init: SMs x resident CTAs)
struct DeviceInfo {
    int device;
    int sm_count;
    size_t total_mem;
};

// the abundance spectrum as a result format (spectrum.cuh): hist[0..hist_len) counters, tail[0..tail_cap) pairs
struct SpecOut {
    unsigned long long* hist;
    uint64_t hist_len;
    kmer_count_pair* tail;
    uint64_t tail_cap;
};

// rows.cu ---------------------------------------------------------------------------------------
// zeroes + fills the row-start mask, flags rows shorter than k (or non-monotone offsets)
void launch_rows_prepare(const uint64_t* d_off, uint64_t n_rows, uint64_t n_bases, int k, uint32_t* d_mask,
                         uint64_t mask_words, DevStatus* d_status, cudaStream_t st);
// row index of the row containing the first base of every tile
// synth.cu: n_rows reads of read_len uniform ACGT bases, rows [first_row, first_row + n_rows) of the table `seed` defines
void launch_synth_reads(const DeviceInfo& di, uint64_t seed, uint64_t first_row, uint64_t n_rows, uint64_t read_len, char* d_seq,
                        uint64_t* d_row_off, cudaStream_t st);
void launch_tile_row_base(const uint64_t* d_off, uint64_t n_rows, uint64_t n_tiles, uint32_t* d_tile_row, cudaStream_t st);

// extract.cu ------------------------------------------------------------------------------------
void launch_extract(const DeviceInfo& di, const ScanArgs& a, const uint32_t* d_tile_row, uint64_t* d_codes,
                    uint64_t capacity, cudaStream_t st);

// count_dense.cu --------------------------------------------------------------------------------
// k <= 13: direct-addressed counters (4^k uint64, zeroed here), then compaction of non-zero bins
// canon: canonical counting -- every window is binned under min(code, reverse complement)
void launch_count_dense(const DeviceInfo& di, const ScanArgs& a, unsigned long long* d_table,
                        kmer_count_pair* d_pairs, uint64_t capacity, cudaStream_t st, bool canon = false);

void launch_dense_table(const DeviceInfo& di, const ScanArgs& a, unsigned long long* d_table, cudaStream_t st, bool canon = false);
void launch_dense_emit(const DeviceInfo& di, const unsigned long long* d_table, int k, uint32_t rank, uint32_t n_ranks,
                       kmer_count_pair* d_pairs, uint64_t capacity, DevStatus* d_status, cudaStream_t st);

// count_hash.cu ---------------------------------------------------------------------------------
// open-addressing table of (code,count) slots in HBM; slots must be filled with 0xFF bytes
void launch_hash_clear(kmer_count_pair* d_slots, uint64_t n_slots, cudaStream_t st);
void launch_count_hash_insert(const DeviceInfo& di, const ScanArgs& a, kmer_count_pair* d_slots, uint64_t n_slots,
                              cudaStream_t st, bool canon = false);
void launch_merge_pairs(const DeviceInfo& di, const kmer_count_pair* d_in, uint64_t n, uint32_t rank, uint32_t n_ranks,
                        kmer_count_pair* d_slots, uint64_t n_slots, DevStatus* d_status, cudaStream_t st);
// appends every occupied slot (+ the k==32 special key) to d_pairs, bumping status->n_distinct
void launch_hash_compact(const DeviceInfo& di, const kmer_count_pair* d_slots, uint64_t n_slots, int k,
                         kmer_count_pair* d_pairs, uint64_t capacity, DevStatus* d_status, cudaStream_t st, int gated = 0);

// spectrum.cu: the spectrum of a table in HBM -- hash table slots (gated: tier 2's, + the k == 32 special key, as
// launch_hash_compact), the dense 4^k counters (bins owned by `rank`), or (k-mer, count) pairs
void launch_hash_spectrum(const DeviceInfo& di, const kmer_count_pair* d_slots, uint64_t n_slots, int k, const SpecOut& o,
                          DevStatus* d_status, cudaStream_t st, int gated = 0);
void launch_dense_spectrum(const DeviceInfo& di, const unsigned long long* d_table, int k, uint32_t rank, uint32_t n_ranks,
                           const SpecOut& o, DevStatus* d_status, cudaStream_t st);
void launch_pairs_spectrum(const DeviceInfo& di, const kmer_count_pair* d_pairs, uint64_t n, const SpecOut& o, DevStatus* d_status,
                           cudaStream_t st);

// count_part.cu --------------------------------------------------------------------------------
struct PartitionPlan {
    uint32_t n_buckets;   // buckets the k-mers are spread over (about 1200 k-mers each)
    uint32_t cap;         // records a bucket region holds
    int w;                // m-mers per minimizer window (4, 6, 8, 9, 12 or 16)
    int m;                // m-mer length (<= 16)
    int recw;             // 64-bit words per super-k-mer record (1: k <= 26, 2: k >= 27)
    int rmax;             // max k-mers per record
    uint64_t spill_cap;   // records the spill list holds
    uint32_t hash_buckets; // range the minimizer hash is scaled to (== n_buckets unless partitioning coarsely)
    int fine_shift;       // bucket = scaled hash >> fine_shift (sharded counting: coarse partitions of 2^fine_shift buckets)
    int even;             // 1: spread the m-mers over the buckets by a second hash (fewer than 30 m-mers per bucket: the load-aware
                          // map of bucket_position() cannot split an m-mer); 0: buckets of equal expected load
};
// canon: the plan of canonical counting (the strand-symmetric minimizer of partition_kernel<.., true>: m may be one base shorter)
PartitionPlan make_partition_plan(uint64_t n_kmers, int k, bool canon = false);
void partition_force_window(int w);   // tests: 0 = automatic
// two write-combining passes (scatter.cuh): column -> n_coarse partitions (one segment per scatter CTA) -> fine buckets
struct ScatterPlan {
    uint32_t n_coarse;   // destinations of the first pass
    uint32_t seg_cap;    // records per (scatter CTA, coarse partition) segment; whole sectors
    uint32_t n_src;      // scatter CTAs = segments per coarse partition
    uint32_t caps;       // staging slots per destination, first pass
    uint32_t caps2;      // staging slots per fine bucket, second pass
};
// Adjusts p (n_buckets = n_coarse << fine_shift) and fills sp; false: the job does not suit the two-pass path (the caller uses
// launch_partition).  Single GPU only: sharded counting scatters into coarse partitions with partition_kernel and splits them
// with refine_staged_kernel on the owner.
bool make_scatter_plan(const DeviceInfo& di, uint64_t n_bases, uint64_t n_kmers, PartitionPlan& p, ScatterPlan& sp);
size_t scatter_seg_bytes(const PartitionPlan& p, const ScatterPlan& sp);
size_t scatter_segfill_bytes(const ScatterPlan& sp);
// d_fill (p.n_buckets words) is zeroed here; afterwards it holds k-mers << 32 | records in the region | poison (bit 31)
void launch_scatter_refine(const DeviceInfo& di, const ScanArgs& a, const PartitionPlan& p, const ScatterPlan& sp, uint32_t* d_segfill,
                           void* d_seg, unsigned long long* d_fill, void* d_recs, void* d_spill, cudaStream_t st,
                           void (*mark)(void*, const char*), void* mark_arg);
size_t partition_record_bytes(const PartitionPlan& p);
size_t partition_spill_bytes(const PartitionPlan& p);
// minimizer partition + per-bucket shared-memory counting (14 <= k <= 32).  Afterwards the host reads
// DevStatus: n_overflow != 0 -> discard and recount (tier 3); n_failed / n_spill != 0 -> run tier 2.
void launch_count_partition(const DeviceInfo& di, const ScanArgs& a, const PartitionPlan& p, unsigned long long* d_fill,
                            void* d_recs, void* d_spill, uint32_t* d_failed_ids, kmer_count_pair* d_pairs, uint64_t capacity,
                            uint64_t* d_uniq, uint64_t uniq_capacity, cudaStream_t st, void (*mark)(void*, const char*), void* mark_arg,
                            const SpecOut* spec = nullptr, bool canon = false);
// a.tile_begin/tile_end: the tiles this launch walks (a column that arrives in pieces); clear_fill = false appends to the regions
void launch_partition(const DeviceInfo& di, const ScanArgs& a, const PartitionPlan& p, unsigned long long* d_fill,
                      void* d_recs, void* d_spill, cudaStream_t st, bool clear_fill = true, bool canon = false);
void launch_bucket_count(const DeviceInfo& di, const PartitionPlan& p, int k, const unsigned long long* d_fill,
                         const void* d_recs, void* d_spill, uint32_t* d_failed_ids, kmer_count_pair* d_pairs, uint64_t capacity,
                         uint64_t* d_uniq, uint64_t uniq_capacity, DevStatus* d_status, cudaStream_t st, uint32_t bucket_begin = 0,
                         uint32_t bucket_end = 0, const SpecOut* spec = nullptr, bool canon = false);
// bucket_begin/bucket_end: the buckets this launch counts (0, 0: all) -- results can leave while later buckets are counted.
// canon: canonical counting (keys canonicalized where the leaf forms them; the plan must come from make_partition_plan(.., true)
// and the records from launch_partition(.., canon = true)).
// d_uniq != nullptr: split result format -- k-mers proven unique on chip are written as bare codes to d_uniq (counted in
// DevStatus::n_unique), everything else as (k-mer, count) pairs.  spec != nullptr: the spectrum result format instead (d_pairs,
// d_uniq unused): every group the leaf counts is binned into spec->hist / spec->tail, nothing is written per group
// Tier 2, stream-ordered: the device itself decides whether the failed buckets / spilled records need it (DevStatus::t2_mode);
// all kernels are always launched and return at once when they are not needed.  d_slots: n_slots (a power of two) table slots;
// if the failed k-mers do not fit, DevStatus::n_overflow is set (the caller recounts in kmer_cuda_dev_finish).
// Also appends the k == 32 special key.
uint64_t tier2_table_slots(uint64_t n_kmers);
void launch_partition_tier2(const DeviceInfo& di, const PartitionPlan& p, int k, const unsigned long long* d_fill,
                            const void* d_recs, const void* d_spill, const uint32_t* d_failed_ids, kmer_count_pair* d_slots,
                            uint64_t n_slots, kmer_count_pair* d_pairs, uint64_t capacity, DevStatus* d_status, cudaStream_t st,
                            void (*mark)(void*, const char*), void* mark_arg, const SpecOut* spec = nullptr, bool canon = false);
// sharded counting, owner side: the coarse partitions received from every source GPU ([src][n_coarse][coarse_cap] records,
// [src][n_coarse] fills) are split into this GPU's fine buckets (p: n_buckets = n_coarse << fine_shift, cap, spill list)
// Source s's segments for THIS owner are src.recs[s] ([n_coarse][coarse_cap] records) and src.fill[s] ([n_coarse] fills): plain
// device pointers, which may point into another GPU's memory (peer access / CUDA IPC) -- the split then pulls the records over
// NVLink itself and no separate exchange step exists.
constexpr int KMER_MAX_SRC = 32;
struct SrcTable {
    const void* recs[KMER_MAX_SRC];
    const unsigned long long* fill[KMER_MAX_SRC];
};
void launch_refine(const DeviceInfo& di, const PartitionPlan& p, int k, int n_src, uint32_t n_coarse, uint32_t coarse_cap,
                   const SrcTable& src, unsigned long long* d_fill, void* d_recs, void* d_spill, DevStatus* d_status, cudaStream_t st);
void launch_append_special(kmer_count_pair* d_pairs, uint64_t capacity, DevStatus* d_status, cudaStream_t st);

// match.cu --------------------------------------------------------------------------------------
struct MatchConst {          // one compiled constant
    uint64_t code;           // equals / starts_with: the literal's code
    uint64_t m0, m1, m2, m3; // contains: for base value b, bit j of m_b set <=> pattern position j (from the
                             // LAST base, j = 0) admits base b          (match(), kmer.h:21-53)
    uint32_t len;            // literal length
    uint32_t pad;
};
// d_ops: optional per-constant op (device array), else `op` for all; any_contains: some constant is a qkmer
void launch_match(const DeviceInfo& di, int op, const int* d_ops, bool any_contains, const uint64_t* d_codes,
                  const uint8_t* d_lens, uint64_t m, int k, const MatchConst* d_consts, uint32_t n_consts,
                  uint32_t* d_bits, uint64_t words_per_row, unsigned long long* d_hits, cudaStream_t st);

// decode.cu -------------------------------------------------------------------------------------
void launch_decode(const DeviceInfo& di, const uint64_t* d_codes, uint64_t n, int k, int with_header, char* d_text,
                   cudaStream_t st);
// uint64 codes -> nbytes-byte little-endian integers (d_out: n * nbytes bytes, 16-byte aligned)
void launch_pack_codes(const DeviceInfo& di, const uint64_t* d_codes, uint64_t n, int nbytes, uint8_t* d_out, cudaStream_t st);
void launch_encode(const DeviceInfo& di, const char* d_text, const uint8_t* d_lens, uint64_t n, int stride,
                   uint64_t* d_codes, DevStatus* d_status, cudaStream_t st);

}  // namespace kmer
