/*
 * kmer_cuda.h -- C ABI of libkmer_cuda.so, the B200 (sm_100a) batch engine for the data-parallel
 * hot path of the PostgreSQL `kmer` extension (NishantSushmakar/kmer-extension).
 *
 * The reference has no batch interface: PostgreSQL calls its C functions once per row / per k-mer
 * through fmgr-V1 (`Datum f(PG_FUNCTION_ARGS)`, kmer.c:84-365).  This header is what new C glue in
 * the extension (see INTEGRATION.md) binds instead, one call per column batch.  Each entry point
 * cites the reference interface it replaces.
 *
 * Conventions
 *   - Plain C linkage, plain pointers and sizes; nothing is thrown or longjmp'ed across the boundary.
 *     Every call returns a kmer_status; kmer_cuda_last_error() gives SQLSTATE / message / detail /
 *     offending row exactly as the reference's ereport() would (kmer.c:33-36,117-119,151-153,
 *     179-181,311-313), so the glue can re-raise it unchanged.
 *   - Rows are a flat text buffer plus offsets: row r is seq[row_off[r] .. row_off[r+1]) -- the
 *     payload of a `dna` varlena (kmer.h:9; 1 byte per base, any case).  row_off[0] must be 0.
 *   - A k-mer is a uint64 code: a=0 c=1 g=2 t=3, first base in the most significant USED bit pair
 *     (code < 4^k).  For equal k, code order == memcmp order of the lower-case text the reference
 *     stores (kmer.c:28-29,124-126) and a prefix is the high bits.  k <= 32 = MAX_KMER_LENGTH
 *     (kmer.h:18).  Columns of mixed-length k-mers carry a parallel uint8 length array.
 *   - There is no CPU fallback.  Without a usable CUDA device every call fails with
 *     KMER_ERR_NO_DEVICE / KMER_ERR_CUDA.
 *   - A context is process-local and NOT thread-safe: one in-flight batch per context.  It creates
 *     its CUDA context lazily inside kmer_cuda_init, so a PostgreSQL backend must call it after
 *     fork(), never in the postmaster.
 */
#ifndef KMER_CUDA_H
#define KMER_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KMER_CUDA_MAX_K 32 /* MAX_KMER_LENGTH, kmer.h:18 */
#define KMER_CUDA_ABI_VERSION 2

typedef enum kmer_status
{
	KMER_OK = 0,
	/* errors the reference raises (same SQLSTATE / text) */
	KMER_ERR_INVALID_DNA = 1,	 /* 22P02 "Invalid DNA Sequence" + detail     validate_sequence kmer.c:31-37 */
	KMER_ERR_KMER_TOO_LONG = 2,	 /* 22001 "KMer Sequence larger than length 32"          kmer_in kmer.c:115-120 */
	KMER_ERR_INVALID_QKMER = 3,	 /* 22P02 "Invalid QKMer Sequence"                      qkmer_in kmer.c:177-182 */
	KMER_ERR_INVALID_K = 4,		 /* 22023 "Invalid KMER Length"                   generate_kmers kmer.c:310-313 */
	KMER_ERR_QKMER_TOO_LONG = 5, /* 22001 "QKMer Sequence larger than length 32"        qkmer_in kmer.c:149-154 */
	/* errors of the engine itself (SQLSTATE XX000 / 53200 in the glue) */
	KMER_ERR_BAD_ARGUMENT = 16,
	KMER_ERR_CUDA = 17,
	KMER_ERR_OOM = 18,
	KMER_ERR_NO_DEVICE = 19,
	KMER_ERR_CAPACITY = 20 /* caller-provided output buffer too small */
} kmer_status;

typedef struct kmer_cuda_error
{
	int status;			 /* kmer_status */
	char sqlstate[6];	 /* "22P02", "22001", "22023", "XX000", "53200" */
	char message[160];	 /* errmsg, verbatim for the reference's errors */
	char detail[160];	 /* errdetail or "" */
	int64_t row;		 /* first offending row of the batch, or -1 */
} kmer_cuda_error;

/* One group of `SELECT kmer, count(*) ... GROUP BY kmer`: the k-mer and its bigint count. */
typedef struct kmer_count_pair
{
	uint64_t code;
	uint64_t count;
} kmer_count_pair;

typedef struct kmer_cuda_ctx kmer_cuda_ctx;

/* predicate selectors for kmer_cuda_*_match (the column is always the `kmer` operand) */
typedef enum kmer_match_op
{
	KMER_OP_EQUALS = 0,		 /* kmer = const          equals(kmer,kmer)        kmer_equals kmer.c:226-245 */
	KMER_OP_STARTS_WITH = 1, /* kmer ^@ const  ==  starts_with(const, kmer)    kmer_starts_with[_op] kmer.c:248-265 */
	KMER_OP_CONTAINS = 2	 /* const::qkmer @> kmer == kmer <@ const          kmer_contains/_containing kmer.c:268-285 */
} kmer_match_op;

/* ---------------------------------------------------------------- lifecycle */

int kmer_cuda_abi_version(void);
/* number of CUDA devices visible, 0 if none / no driver */
int kmer_cuda_device_count(void);
/* Creates a context on `device` (creates the CUDA primary context lazily, here). */
int kmer_cuda_init(kmer_cuda_ctx **ctx, int device);
void kmer_cuda_shutdown(kmer_cuda_ctx *ctx);
/* Error record of the last failing call on ctx (ctx may be NULL: error of the last failed init). */
const kmer_cuda_error *kmer_cuda_last_error(const kmer_cuda_ctx *ctx);
/* Frees a result buffer returned by a kmer_cuda_submit_* call (pinned host memory). */
void kmer_cuda_release(kmer_cuda_ctx *ctx, void *result);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
uint64_t kmer_cuda_launch_count(const kmer_cuda_ctx *ctx);

/* Test hook (process-wide, not for production use): forces the minimizer window of the partition counter (4/6/8 for k <= 26,
 * 8/12/16 for k >= 27; 0 = automatic) so that the parity tests cover every window the kernels are built for. */
void kmer_cuda_test_force_window(int w);

/* Phase timing for benchmarks: when on, CUDA events bracket every kernel phase of a dev_* call;
 * after kmer_cuda_dev_finish(), kmer_cuda_get_phases() returns the phase names (static strings)
 * and their device durations in ms.  Returns the number of phases of the last finished call. */
void kmer_cuda_set_profiling(kmer_cuda_ctx *ctx, int on);
int kmer_cuda_get_phases(const kmer_cuda_ctx *ctx, const char **names, float *ms, int capacity);

/* ---------------------------------------------------------------- host-buffer batch submit
 * Inputs are caller-owned host memory (pageable or pinned); results are library-owned pinned host
 * buffers, valid until kmer_cuda_release().  Calls block until the result is complete. */

/* Replaces one generate_kmers SRF scan per row (kmer.c:289-351) for a whole column:
 * (*codes)[0..*n_kmers) = every window of every row, rows in order, positions in order.
 * Any row shorter than k, or k outside 1..32, fails the batch with KMER_ERR_INVALID_K
 * (kmer.c:310-313); any byte outside ACGTacgt fails it with KMER_ERR_INVALID_DNA (kmer.c:20-41).
 * The first offending row decides, as in a sequential scan. */
int kmer_cuda_submit_extract(kmer_cuda_ctx *ctx, const char *seq, const uint64_t *row_off, uint64_t n_rows,
							 int k, uint64_t **codes, uint64_t *n_kmers);

/* Replaces `SELECT kmer, count(*) FROM (SELECT generate_kmers(dna,k) ...) GROUP BY kmer`
 * (generate_kmers kmer.c:289-351 + HashAggregate over kmer_hash kmer.c:353-365 / kmer_equals
 * kmer.c:226-245): (*pairs)[0..*n_distinct) in unspecified order, like a hash aggregate's output.
 * Same error behaviour as kmer_cuda_submit_extract.  *n_kmers = total windows counted. */
int kmer_cuda_submit_count(kmer_cuda_ctx *ctx, const char *seq, const uint64_t *row_off, uint64_t n_rows,
						   int k, kmer_count_pair **pairs, uint64_t *n_distinct, uint64_t *n_kmers);

/* The same GROUP BY in the split result format: a group whose count is 1 is returned as its bare code,
 * (*uniq_codes)[0..*n_unique); every other group -- and any count-1 group the device did not prove unique on chip --
 * as a pair, (*pairs)[0..*n_pairs).  The union of the two is exactly kmer_cuda_submit_count()'s table; no k-mer is in
 * both.  On mostly distinct k-mers (k >= 14 over unassembled reads) this halves the bytes that cross PCIe: 8 instead
 * of 16 per group.  Both buffers are released separately with kmer_cuda_release(). */
int kmer_cuda_submit_count_split(kmer_cuda_ctx *ctx, const char *seq, const uint64_t *row_off, uint64_t n_rows, int k,
								 uint64_t **uniq_codes, uint64_t *n_unique, kmer_count_pair **pairs, uint64_t *n_pairs,
								 uint64_t *n_kmers);

/* The split format with the bare codes packed for transport: (*uniq_packed) holds *n_unique little-endian integers
 * of *code_bytes = ceil(2k/8) bytes each (6 at k=21 instead of 8; the reference's own kmer datum is k+1 = 22 bytes),
 * code i at byte offset i * *code_bytes.  Everything else as kmer_cuda_submit_count_split. */
int kmer_cuda_submit_count_packed(kmer_cuda_ctx *ctx, const char *seq, const uint64_t *row_off, uint64_t n_rows, int k,
								  uint8_t **uniq_packed, uint64_t *n_unique, int *code_bytes, kmer_count_pair **pairs,
								  uint64_t *n_pairs, uint64_t *n_kmers);

/* The k-mer abundance spectrum (count of counts) of the same GROUP BY -- what `jellyfish histo`, KAT and GenomeScope work from:
 *   SELECT cnt AS count, count(*) AS kmers
 *   FROM (SELECT count(*) AS cnt FROM reads r, generate_kmers(r.dna, k) AS g(kmer) GROUP BY g.kmer) s GROUP BY cnt
 * (*hist)[c], 1 <= c < hist_len (>= 2): number of distinct k-mers counted exactly c times; (*hist)[0] = 0.  Every group whose
 * count is >= hist_len comes back whole in (*tail)[0..*n_tail), in unspecified order (the high-copy k-mers themselves), so
 * the spectrum is exact for any count.  The groups are binned on the device: no buffer of the table's size exists on either
 * side of PCIe.  Same errors as kmer_cuda_submit_count.  Both results are released with kmer_cuda_release(). */
int kmer_cuda_submit_count_spectrum(kmer_cuda_ctx *ctx, const char *seq, const uint64_t *row_off, uint64_t n_rows, int k,
									uint64_t hist_len, uint64_t **hist, kmer_count_pair **tail, uint64_t *n_tail,
									uint64_t *n_kmers);

/* Canonical k-mer counting: a k-mer and its reverse complement are one group (what `jellyfish count -C`, KMC and Gerbil count by
 * default, and the spectrum GenomeScope expects: reads come from both strands).  rc(x) complements every base (a<->t, c<->g) and
 * reverses their order; canon(x) = min(x, rc(x)), which is also the smaller of the two lower-case texts.  One group per value of
 * canon over all windows of all rows, counted over windows of either orientation; equal to the stock SQL
 *   SELECT least(g.kmer::text COLLATE "C", reverse(translate(g.kmer::text, 'acgt', 'tgca')))::kmer AS kmer, count(*)
 *   FROM reads r, generate_kmers(r.dna, k) AS g(kmer) GROUP BY 1
 * Errors and the offending row are exactly those of kmer_cuda_submit_count.  Every code returned is canonical; at k = 32 the
 * all-t and all-a windows are one group with code 0.  The strand-specific calls are unchanged (they are the reference's
 * contract); canonical counting is a separate set of entry points, never a mode left on a context.  Not covered: sharded
 * counting, the packed format, extract.
 * uniq_codes == NULL: every group in (*pairs)[0..*n_pairs) (kmer_cuda_submit_count's format); else the split format of
 * kmer_cuda_submit_count_split.  Results are released with kmer_cuda_release(). */
int kmer_cuda_submit_count_canonical(kmer_cuda_ctx *ctx, const char *seq, const uint64_t *row_off, uint64_t n_rows, int k,
									 uint64_t **uniq_codes, uint64_t *n_unique, kmer_count_pair **pairs, uint64_t *n_pairs,
									 uint64_t *n_kmers);
/* The abundance spectrum of the canonical GROUP BY: the contract of kmer_cuda_submit_count_spectrum. */
int kmer_cuda_submit_count_canonical_spectrum(kmer_cuda_ctx *ctx, const char *seq, const uint64_t *row_off, uint64_t n_rows,
											  int k, uint64_t hist_len, uint64_t **hist, kmer_count_pair **tail, uint64_t *n_tail,
											  uint64_t *n_kmers);

/* Replaces per-row calls of kmer_equals / kmer_starts_with[_op] / kmer_contains / kmer_containing
 * (kmer.c:226-285) over a column of m k-mers against n_consts constants given as text:
 *   KMER_OP_EQUALS, KMER_OP_STARTS_WITH : constants are kmer literals   (kmer_in rules, kmer.c:109-129)
 *   KMER_OP_CONTAINS                    : constants are qkmer literals  (qkmer_in rules, kmer.c:141-190)
 * ops == NULL: every constant uses `op`; else ops[c] (a kmer_match_op) selects the predicate of
 * constant c, so that e.g. an equals and a starts_with filter share one pass over the column.
 * lens == NULL: every k-mer has length k; else lens[i] (0..32) is the length of codes[i].
 * Result: bit matrix, row c = constant c, (*bits)[c * words_per_row + (i >> 5)] bit (i & 31) is the
 * boolean the reference returns for (const c, kmer i); words_per_row = ceil(m / 32), returned in
 * *words_per_row; (*hits)[c] = number of set bits of row c. */
int kmer_cuda_submit_match(kmer_cuda_ctx *ctx, int op, const int *ops, const uint64_t *codes, const uint8_t *lens,
						   uint64_t m, int k, const char *const *consts, uint32_t n_consts, uint32_t **bits,
						   uint64_t *words_per_row, uint64_t **hits);

/* Text of a column of k-mers as the reference stores it: lower-case ASCII, kmer_out kmer.c:131-138.
 * with_header == 0: (*text) is n*k bytes.  with_header != 0: n*(k+1) bytes, each k-mer prefixed by
 * its 1-byte short varlena header ((k+1)<<1|1, SET_VARSIZE_SHORT kmer.c:341-342), i.e. the exact
 * bytes of the `kmer` datums generate_kmers would have palloc'ed (little-endian servers). */
int kmer_cuda_submit_decode(kmer_cuda_ctx *ctx, const uint64_t *codes, uint64_t n, int k, int with_header,
							char **text);

/* Parses a column of k-mer texts (n fixed-stride records of `stride` bytes, lens[i] bytes used,
 * lens == NULL: all `stride`) into codes: batched kmer_in (kmer.c:109-129). */
int kmer_cuda_submit_encode(kmer_cuda_ctx *ctx, const char *text, const uint8_t *lens, uint64_t n, int stride,
							uint64_t **codes);

/* ---------------------------------------------------------------- device-resident API
 * Same operations on buffers already in HBM (device pointers), asynchronous on `stream`
 * (a cudaStream_t passed as void*; NULL = the CUDA default stream).  Used for resident-data
 * benchmarking and by the multi-GPU pipeline, which keeps shards in HBM between steps.
 * d_seq must be 16-byte aligned and readable up to the next multiple of 16 bytes.
 * Results that are counts land in the struct filled by kmer_cuda_dev_finish(), which synchronises
 * the stream and reports input errors found by the kernels. */

typedef struct kmer_dev_result
{
	uint64_t n_kmers;	 /* windows produced / counted by the last extract or count */
	uint64_t n_distinct; /* groups written by the last count */
	uint64_t n_overflow; /* != 0: the partition counter gave up and the batch was recounted through the
						  * global hash table (highly repetitive input); diagnostics only */
	uint64_t n_tier2;	 /* k-mers of buckets that did not fit on chip and were counted by the tier-2
						  * kernel instead; diagnostics only */
	uint64_t n_unique;	 /* kmer_cuda_dev_count_split: bare codes written (n_distinct counts the pairs only) */
} kmer_dev_result;

int kmer_cuda_dev_extract(kmer_cuda_ctx *ctx, const char *d_seq, uint64_t n_bases, const uint64_t *d_row_off,
						  uint64_t n_rows, int k, uint64_t *d_codes, uint64_t codes_capacity, void *stream);

/* algo: 0 = automatic, 1 = dense table (k small), 2 = global hash table, 3 = minimizer partition,
 * 4 = minimizer partition through two write-combining passes (experimental; falls back to 3 when the job does not suit it) */
int kmer_cuda_dev_count(kmer_cuda_ctx *ctx, const char *d_seq, uint64_t n_bases, const uint64_t *d_row_off,
						uint64_t n_rows, int k, kmer_count_pair *d_pairs, uint64_t pairs_capacity, int algo,
						void *stream);

/* Split result format (see kmer_cuda_submit_count_split): unique k-mers as bare codes in d_uniq, the rest as pairs. */
int kmer_cuda_dev_count_split(kmer_cuda_ctx *ctx, const char *d_seq, uint64_t n_bases, const uint64_t *d_row_off,
							  uint64_t n_rows, int k, uint64_t *d_uniq, uint64_t uniq_capacity, kmer_count_pair *d_pairs,
							  uint64_t pairs_capacity, void *stream);

/* Spectrum result format (see kmer_cuda_submit_count_spectrum): d_hist[0..hist_len) is overwritten whole (hist_len >= 2), the
 * groups with count >= hist_len are written to d_tail; floor(n_windows / hist_len) entries always suffice, fewer than needed fail
 * with KMER_ERR_CAPACITY.  kmer_cuda_dev_finish() reports n_kmers = windows counted, n_distinct = tail entries written,
 * n_tier2 / n_overflow as for kmer_cuda_dev_count, n_unique = 0.  algo as kmer_cuda_dev_count (1 = dense, 2 = hash, 3 / 4 =
 * partition; 0 = dense for k <= 13, partition for k >= 14); same errors. */
int kmer_cuda_dev_count_spectrum(kmer_cuda_ctx *ctx, const char *d_seq, uint64_t n_bases, const uint64_t *d_row_off,
								 uint64_t n_rows, int k, uint64_t *d_hist, uint64_t hist_len, kmer_count_pair *d_tail,
								 uint64_t tail_capacity, int algo, void *stream);
/* Canonical counting (see kmer_cuda_submit_count_canonical) on device buffers.  d_uniq == NULL: every group as a pair in d_pairs
 * (kmer_cuda_dev_count's format); else the split format of kmer_cuda_dev_count_split.  algo as kmer_cuda_dev_count, except that
 * 4 runs as 3 (the two-pass partition has no canonical minimizer). */
int kmer_cuda_dev_count_canonical(kmer_cuda_ctx *ctx, const char *d_seq, uint64_t n_bases, const uint64_t *d_row_off,
								  uint64_t n_rows, int k, uint64_t *d_uniq, uint64_t uniq_capacity, kmer_count_pair *d_pairs,
								  uint64_t pairs_capacity, int algo, void *stream);
/* The spectrum of the canonical GROUP BY: the arguments, outputs and finish() report of kmer_cuda_dev_count_spectrum. */
int kmer_cuda_dev_count_canonical_spectrum(kmer_cuda_ctx *ctx, const char *d_seq, uint64_t n_bases, const uint64_t *d_row_off,
										   uint64_t n_rows, int k, uint64_t *d_hist, uint64_t hist_len, kmer_count_pair *d_tail,
										   uint64_t tail_capacity, int algo, void *stream);
/* The spectrum of a (k-mer, count) table already in HBM, d_pairs[0..n): same outputs and finish() report. */
int kmer_cuda_dev_pairs_spectrum(kmer_cuda_ctx *ctx, const kmer_count_pair *d_pairs, uint64_t n, uint64_t *d_hist,
								 uint64_t hist_len, kmer_count_pair *d_tail, uint64_t tail_capacity, void *stream);

/* consts / ops are HOST arrays (they are compiled to masks on the host); d_* are device pointers.
 * d_bits: n_consts * ceil(m/32) words; d_hits: n_consts counters. */
int kmer_cuda_dev_match(kmer_cuda_ctx *ctx, int op, const int *ops, const uint64_t *d_codes, const uint8_t *d_lens,
						uint64_t m, int k, const char *const *consts, uint32_t n_consts, uint32_t *d_bits,
						uint64_t *d_hits, void *stream);

int kmer_cuda_dev_decode(kmer_cuda_ctx *ctx, const uint64_t *d_codes, uint64_t n, int k, int with_header,
						 char *d_text, void *stream);

/* Transport form of a column of bare codes (kmer_cuda_submit_count_packed): n little-endian integers of ceil(2k/8) bytes each,
 * d_packed 16-byte aligned with room for n * ceil(2k/8) bytes.  Stream-ordered, no finish needed. */
int kmer_cuda_dev_pack_codes(kmer_cuda_ctx *ctx, const uint64_t *d_codes, uint64_t n, int k, uint8_t *d_packed, void *stream);

int kmer_cuda_dev_finish(kmer_cuda_ctx *ctx, void *stream, kmer_dev_result *result);

/* ---------------------------------------------------------------- sharded counting (one process per GPU)
 * Counting shards by row.  Every GPU partitions ITS rows' k-mers (as super-k-mer records) into the same global
 * set of coarse minimizer partitions; partition p is owned by GPU p / buckets_per_rank; one all-to-all moves
 * every (partition, source) segment to its owner; the owner splits its partitions into 2^fine_shift fine buckets
 * each and counts those on chip.  Identical k-mers share a minimizer, hence a partition, hence an owner: the
 * per-GPU results are disjoint and the GROUP BY result is their concatenation.  The number of regions a source
 * GPU scatters into (n_buckets) does not grow with the size of the job, only their size does.
 * The library does no communication itself; the caller runs the exchange (NCCL all-to-all with equal splits in
 * bench.py / sharded.py; ncclSend/ncclRecv from C):
 *
 *   kmer_cuda_shard_plan()            same arguments on every rank -> same plan
 *   kmer_cuda_dev_shard_partition()   rows -> send_recs [n_buckets][cap] records, send_fill [n_buckets]
 *   all-to-all(send_recs, recs_bytes_per_peer)  and  all-to-all(send_fill, fill_bytes_per_peer)
 *   kmer_cuda_dev_shard_count()       recv_recs [n_ranks * chunks_per_rank][buckets_per_rank][cap], recv_fill likewise
 *                                     -> this rank's (k-mer, count) pairs
 * 14 <= k <= 32.  (Smaller k: kmer_cuda_dev_dense_table + all-reduce + kmer_cuda_dev_dense_emit.) */
typedef struct kmer_shard_plan
{
	uint32_t n_ranks;
	uint32_t n_buckets;		   /* coarse partitions, global; = n_ranks * buckets_per_rank */
	uint32_t buckets_per_rank;
	uint32_t cap;			   /* records per (partition, source GPU) segment; even */
	int32_t k;
	int32_t rec_bytes;		   /* 8 (k <= 26) or 16 */
	uint64_t recs_bytes_per_peer; /* buckets_per_rank * cap * rec_bytes */
	uint64_t fill_bytes_per_peer; /* buckets_per_rank * 8 */
	int32_t w, m, recw, rmax;  /* minimizer window / m-mer length / record words / max k-mers per record */
	uint32_t fine_shift;	   /* every partition is split into 2^fine_shift fine buckets by its owner */
	uint32_t fine_cap;		   /* records per fine bucket region (owner side workspace) */
	uint32_t chunks_per_rank;  /* segments per source GPU (kmer_cuda_shard_plan_chunked), 1 otherwise */
	uint32_t even_spread;	   /* 1: few distinct m-mers per bucket (short k, huge job): m-mers are spread by a second hash */
} kmer_shard_plan;

int kmer_cuda_shard_plan(uint64_t total_kmers_all_ranks, int k, uint32_t n_ranks, kmer_shard_plan *plan);
/* The same plan when every GPU partitions its rows in `chunks_per_rank` pieces, each into its own send buffer
 * ([n_buckets][cap], cap sized for a piece), so that the exchange of piece i overlaps the partition pass of piece i+1.
 * kmer_cuda_dev_shard_count() then takes recv_recs [chunks_per_rank * n_ranks][buckets_per_rank][cap] (segments in any
 * order) and recv_fill likewise. */
int kmer_cuda_shard_plan_chunked(uint64_t total_kmers_all_ranks, int k, uint32_t n_ranks, uint32_t chunks_per_rank,
								 kmer_shard_plan *plan);
/* Fails with KMER_ERR_CAPACITY (reported by kmer_cuda_dev_finish) if a segment overflows: input too
 * repetitive for this path; nothing may be used then. */
int kmer_cuda_dev_shard_partition(kmer_cuda_ctx *ctx, const char *d_seq, uint64_t n_bases, const uint64_t *d_row_off,
								  uint64_t n_rows, const kmer_shard_plan *plan, void *d_send_recs,
								  uint64_t *d_send_fill, void *stream);
int kmer_cuda_dev_shard_count(kmer_cuda_ctx *ctx, const kmer_shard_plan *plan, const void *d_recv_recs,
							  const uint64_t *d_recv_fill, kmer_count_pair *d_pairs, uint64_t pairs_capacity,
							  void *stream);
/* The same with this rank's share in the split result format (kmer_cuda_dev_count_split). */
int kmer_cuda_dev_shard_count_split(kmer_cuda_ctx *ctx, const kmer_shard_plan *plan, const void *d_recv_recs,
									const uint64_t *d_recv_fill, uint64_t *d_uniq, uint64_t uniq_capacity,
									kmer_count_pair *d_pairs, uint64_t pairs_capacity, void *stream);
/* The exchange fused into the count: this rank reads source s's segments where they lie.  src_recs[s] / src_fill[s]
 * (s < n_ranks * chunks_per_rank; host arrays of device pointers) point at source s's send buffers AT THIS RANK'S
 * BLOCK -- (char *)send_recs_s + rank * plan->recs_bytes_per_peer and send_fill_s + rank * plan->buckets_per_rank --
 * in this GPU's memory or, over NVLink, in another GPU's (peer access inside one process; kmer_cuda_ipc_open across
 * processes).  No all-to-all and no receive buffers: the split kernel pulls the records itself.  The caller orders the
 * call behind every source's kmer_cuda_dev_shard_partition (an event, or any collective enqueued on `stream`) and
 * keeps the sources from overwriting their send buffers until this rank's kmer_cuda_dev_finish has returned.
 * d_uniq may be NULL (pairs only), else the split result format. */
int kmer_cuda_dev_shard_count_peers(kmer_cuda_ctx *ctx, const kmer_shard_plan *plan, const void *const *src_recs,
									const uint64_t *const *src_fill, uint64_t *d_uniq, uint64_t uniq_capacity,
									kmer_count_pair *d_pairs, uint64_t pairs_capacity, void *stream);
/* This rank's share of sharded counting in the spectrum result format (kmer_cuda_dev_count_spectrum), sources given as in
 * kmer_cuda_dev_shard_count_peers.  After the all-to-all, the receive buffers are passed in the same form:
 * src_recs[s] = (char *)recv_recs + s * plan->recs_bytes_per_peer, src_fill[s] = recv_fill + s * plan->buckets_per_rank.
 * The owners' groups are disjoint: the ranks' histograms sum, and their tails concatenate, to the spectrum of all rows. */
int kmer_cuda_dev_shard_count_spectrum(kmer_cuda_ctx *ctx, const kmer_shard_plan *plan, const void *const *src_recs,
									   const uint64_t *const *src_fill, uint64_t *d_hist, uint64_t hist_len,
									   kmer_count_pair *d_tail, uint64_t tail_capacity, void *stream);
/* CUDA IPC for one-process-per-GPU hosts: export names the cudaMalloc ALLOCATION d_ptr lies in (handle64: 64 bytes to
 * send to the peers) and d_ptr's offset inside it; open maps a peer's allocation into this process (enabling peer
 * access from ctx's GPU) and returns its base; close unmaps it.  A handle can be open once per process. */
int kmer_cuda_ipc_export(kmer_cuda_ctx *ctx, const void *d_ptr, void *handle64, uint64_t *offset);
int kmer_cuda_ipc_open(kmer_cuda_ctx *ctx, const void *handle64, void **d_base);
int kmer_cuda_ipc_close(kmer_cuda_ctx *ctx, void *d_base);
/* k <= 13: the dense 4^k table of uint64 counters of this rank's rows (to be summed across ranks),
 * and the emission of the bins owned by `rank` (bin % n_ranks == rank) of a summed table. */
int kmer_cuda_dev_dense_table(kmer_cuda_ctx *ctx, const char *d_seq, uint64_t n_bases, const uint64_t *d_row_off,
							  uint64_t n_rows, int k, uint64_t *d_table, void *stream);
int kmer_cuda_dev_dense_emit(kmer_cuda_ctx *ctx, const uint64_t *d_table, int k, uint32_t rank, uint32_t n_ranks,
							 kmer_count_pair *d_pairs, uint64_t pairs_capacity, void *stream);

/* Exact fallback of sharded counting for input the minimizer exchange refuses (KMER_ERR_CAPACITY: a segment or the spill
 * list overflowed -- highly repetitive rows): every rank counts ITS rows with kmer_cuda_dev_count (exact on any input), then
 * the per-rank tables are merged by owner: owner(k-mer) = hash(k-mer) % n_ranks.  Every rank sees every rank's table in turn
 * (a broadcast by the caller) and adds the groups it owns:
 *   kmer_cuda_dev_merge_begin(max_groups)            table for at most max_groups groups owned by this rank
 *   kmer_cuda_dev_merge_add(table, n, rank, n_ranks) once per source table
 *   kmer_cuda_dev_merge_emit(k, pairs, capacity)     this rank's groups; kmer_cuda_dev_finish() reports n_distinct / n_kmers
 * The per-rank results are disjoint, their union is the GROUP BY of all rows (HashAggregate never refuses input:
 * kmer-tests.sql:1208-1213). */
int kmer_cuda_dev_merge_begin(kmer_cuda_ctx *ctx, uint64_t max_groups, void *stream);
int kmer_cuda_dev_merge_add(kmer_cuda_ctx *ctx, const kmer_count_pair *d_pairs, uint64_t n, uint32_t rank, uint32_t n_ranks,
							void *stream);
int kmer_cuda_dev_merge_emit(kmer_cuda_ctx *ctx, int k, kmer_count_pair *d_pairs, uint64_t pairs_capacity, void *stream);

/* ---------------------------------------------------------------- several GPUs, one process (no Python, no NCCL)
 * What the PostgreSQL glue links when the box has more than one GPU ("Host code stays C ... calls CUDA through a thin C-ABI
 * layer"): the device list is given once; kmer_cuda_multi_submit_count splits the rows evenly over the devices, runs the
 * sharded count above with the exchange done as peer copies over NVLink, and hands back ONE TABLE PER DEVICE:
 * pairs[d][0 .. n_distinct[d]) for d < kmer_cuda_multi_device_count().  The tables are disjoint, their union is the result of
 * `SELECT kmer, count(*) ... GROUP BY kmer` over all rows (kmer.c:289-351 + kmer_hash_ops).  Same errors as
 * kmer_cuda_submit_count, the first offending row of the whole batch decides.  Input the minimizer exchange refuses (highly
 * repetitive rows) and k <= 13 are counted per device and merged by owner, reading the peers' tables over NVLink.
 * Each table is released with kmer_cuda_multi_release(m, d, pairs[d]). */
typedef struct kmer_cuda_multi kmer_cuda_multi;
int kmer_cuda_init_multi(kmer_cuda_multi **m, const int *devices, int n_devices);
void kmer_cuda_shutdown_multi(kmer_cuda_multi *m);
int kmer_cuda_multi_device_count(const kmer_cuda_multi *m);
const kmer_cuda_error *kmer_cuda_multi_last_error(const kmer_cuda_multi *m);
int kmer_cuda_multi_submit_count(kmer_cuda_multi *m, const char *seq, const uint64_t *row_off, uint64_t n_rows, int k,
								 kmer_count_pair **pairs, uint64_t *n_distinct, uint64_t *n_kmers);
void kmer_cuda_multi_release(kmer_cuda_multi *m, int device_index, void *result);
/* kmer_cuda_submit_match on every device of the handle (kmer_equals / kmer_starts_with[_op] / kmer_contains / kmer_containing,
 * kmer.c:226-285, are independent per k-mer: the column is sharded, the constants are replicated, nothing is exchanged).
 * The column is cut on multiples of 32 k-mers, device d matches its slice, and its words of every row are copied straight to
 * their place in ONE bit matrix with the layout of kmer_cuda_submit_match (row c = constant c, words_per_row = ceil(m/32));
 * (*hits)[c] is the sum over the devices.  Same errors as kmer_cuda_submit_match (a bad constant: row = its index).
 * Both results belong to device 0 of the handle: kmer_cuda_multi_release(m, 0, *bits) / (m, 0, *hits). */
int kmer_cuda_multi_submit_match(kmer_cuda_multi *m, int op, const int *ops, const uint64_t *codes, const uint8_t *lens,
								 uint64_t n_kmers, int k, const char *const *consts, uint32_t n_consts, uint32_t **bits,
								 uint64_t *words_per_row, uint64_t **hits);

/* Benchmark inputs generated in HBM (SURVEY 8d2: the reference's data_generator.py:4-11 distribution -- bases i.i.d. uniform
 * over ACGT, upper case -- made seeded and shape-parameterised): rows [first_row, first_row + n_rows) of the table of
 * read_len-base reads that `seed` defines; base g of the table depends on (seed, g) only, so the ranks of a sharded run each
 * generate their own row range of ONE table.  d_seq: n_rows*read_len bytes rounded up to 16 (+64 bytes of padding as every
 * dev_* call wants), 16-byte aligned; d_row_off: n_rows+1 offsets, starting at 0.  Asynchronous on `stream`.
 * Restated in numpy by kmer-extension_b200/datagen.py: synth_reads_counter. */
int kmer_cuda_dev_synth_reads(kmer_cuda_ctx *ctx, uint64_t seed, uint64_t first_row, uint64_t n_rows, uint64_t read_len,
							  char *d_seq, uint64_t *d_row_off, void *stream);

/* Upper bound of the number of k-mers (= groups) a batch can produce: n_bases - n_rows*(k-1). */
uint64_t kmer_cuda_max_kmers(uint64_t n_bases, uint64_t n_rows, int k);

#ifdef __cplusplus
}
#endif
#endif /* KMER_CUDA_H */
