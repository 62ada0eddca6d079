/*
 * kmer_gpu.c -- C glue a maintainer adds NEXT TO the reference's kmer.c (same MODULE_big), binding
 * libkmer_cuda.so through include/kmer_cuda.h.  The existing SQL surface (kmer--1.0.0.sql) is not
 * touched; these functions are additive.  Compiles against PostgreSQL's headers, and -- for the
 * compile check in this repository, which has no PostgreSQL -- against oracle/pgshim.
 *
 *   kmer_gpu_count_datums()  : GROUP BY kmer / count(*) over generate_kmers(dna, k) for a batch of `dna`
 *                              datums, replacing one generate_kmers SRF scan per row (kmer.c:289-351) and
 *                              the HashAggregate over kmer_hash / kmer_equals (kmer.c:226-245,353-365).
 *   kmer_gpu_match_datums()  : equals / starts_with / contains over a batch of `kmer` datums against one
 *                              constant, replacing per-row kmer_equals / kmer_starts_with / kmer_contains
 *                              calls (kmer.c:226-285).
 *   kmer_gpu_spectrum_datums(): the k-mer abundance spectrum (count of counts) of that GROUP BY, binned on the GPU:
 *                              (count, number of k-mers with that count) rows, ascending by count.
 *   kmer_gpu_canonical_count_datums() / kmer_gpu_canonical_spectrum_datums(): the same for canonical k-mers (a k-mer and
 *                              its reverse complement are one group, keyed by the smaller of the two).
 *
 * Results are palloc'ed in the caller's memory context, exactly like the reference's functions
 * (kmer.c:92,124,341); `kmer` results carry the 1-byte short varlena header generate_kmers writes
 * (SET_VARSIZE_SHORT, kmer.c:341-342).  Errors are re-raised with the reference's own SQLSTATE and
 * text (kmer.c:33-36,117-119,151-153,179-181,311-313).
 *
 * CUDA must not be initialised in the postmaster: the context is created lazily, on first use, in
 * the backend (or parallel worker) process, i.e. after fork().
 */
#include "postgres.h"
#include "fmgr.h"
#include "funcapi.h"
#include "utils/array.h"
#include "kmer_cuda.h"

/*
 * SQL surface a maintainer adds next to kmer--1.0.0.sql (additive; nothing existing changes):
 *
 *   CREATE FUNCTION kmer_gpu_counts(dna[], integer) RETURNS TABLE (kmer kmer, count bigint)
 *       AS 'MODULE_PATHNAME', 'kmer_gpu_counts' LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;
 *       -- SELECT * FROM kmer_gpu_counts(ARRAY(SELECT dna FROM reads), 21)
 *       --   ==  SELECT k.kmer, count(*) FROM reads r, generate_kmers(r.dna, 21) AS k(kmer) GROUP BY k.kmer
 *   CREATE FUNCTION kmer_gpu_match(kmer[], text, integer) RETURNS SETOF boolean
 *       AS 'MODULE_PATHNAME', 'kmer_gpu_match' LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;
 *       -- element i: op 0 kmer[i] = $2 ; op 1 kmer[i] ^@ $2 ; op 2 $2::qkmer @> kmer[i]
 *   CREATE FUNCTION kmer_gpu_count_spectrum(dna[], integer) RETURNS TABLE (count bigint, kmers bigint)
 *       AS 'MODULE_PATHNAME', 'kmer_gpu_count_spectrum' LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;
 *       -- SELECT * FROM kmer_gpu_count_spectrum(ARRAY(SELECT dna FROM reads), 21)
 *       --   ==  SELECT cnt AS count, count(*) AS kmers
 *       --       FROM (SELECT count(*) AS cnt FROM reads r, generate_kmers(r.dna, 21) AS g(kmer) GROUP BY g.kmer) s
 *       --       GROUP BY cnt ORDER BY cnt
 *   CREATE FUNCTION kmer_gpu_canonical_counts(dna[], integer) RETURNS TABLE (kmer kmer, count bigint)
 *       AS 'MODULE_PATHNAME', 'kmer_gpu_canonical_counts' LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;
 *   CREATE FUNCTION kmer_gpu_canonical_count_spectrum(dna[], integer) RETURNS TABLE (count bigint, kmers bigint)
 *       AS 'MODULE_PATHNAME', 'kmer_gpu_canonical_count_spectrum' LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;
 *       -- the two above with the k-mer least(kmer::text COLLATE "C", reverse(translate(kmer::text, 'acgt', 'tgca')))::kmer
 */


static kmer_cuda_ctx *gpu_ctx = NULL; /* one per backend process */

static void
kmer_gpu_raise(const kmer_cuda_error *e)
{
	int code;

	switch (e->status)
	{
	case KMER_ERR_INVALID_DNA:
	case KMER_ERR_INVALID_QKMER:
		code = ERRCODE_INVALID_TEXT_REPRESENTATION; /* 22P02 */
		break;
	case KMER_ERR_KMER_TOO_LONG:
	case KMER_ERR_QKMER_TOO_LONG:
		code = ERRCODE_STRING_DATA_RIGHT_TRUNCATION; /* 22001 */
		break;
	case KMER_ERR_INVALID_K:
		code = ERRCODE_INVALID_PARAMETER_VALUE; /* 22023 */
		break;
	case KMER_ERR_OOM:
		code = ERRCODE_OUT_OF_MEMORY;
		break;
	default:
		code = ERRCODE_INTERNAL_ERROR;
	}
	if (e->detail[0])
		ereport(ERROR, (errcode(code), errmsg("%s", e->message), errdetail("%s", e->detail)));
	else
		ereport(ERROR, (errcode(code), errmsg("%s", e->message)));
}

static kmer_cuda_ctx *
kmer_gpu_context(void)
{
	if (gpu_ctx == NULL)
	{
		if (kmer_cuda_init(&gpu_ctx, 0) != KMER_OK) /* device choice: a GUC in a real build */
			kmer_gpu_raise(kmer_cuda_last_error(NULL));
	}
	return gpu_ctx;
}

/*
 * dnas[0..n) are detoasted `dna` datums (PG_DETOAST_DATUM in the caller).  On return *kmers is an array
 * of *n_groups `kmer` datums (short-header varlenas) and *counts their bigint counts.
 */
static void
count_datums(struct varlena **dnas, uint64_t n, int k, bool canonical, struct varlena ***kmers, int64_t **counts,
			 uint64_t *n_groups)
{
	kmer_cuda_ctx *ctx = kmer_gpu_context();
	uint64_t *off = (uint64_t *) palloc((n + 1) * sizeof(uint64_t));
	uint64_t total = 0, i, n_kmers = 0, d = 0, n_uniq = 0, n_pairs = 0;
	uint64_t *uniq = NULL;
	char *flat, *text = NULL;
	kmer_count_pair *pairs = NULL;
	uint64_t *codes;

	off[0] = 0;
	for (i = 0; i < n; i++)
	{
		total += (uint64_t) VARSIZE_ANY_EXHDR(dnas[i]);
		off[i + 1] = total;
	}
	flat = (char *) palloc(total + 16);
	for (i = 0; i < n; i++)
		memcpy(flat + off[i], VARDATA_ANY(dnas[i]), (size_t) (off[i + 1] - off[i]));

	/* split result format: groups with count 1 come back as bare codes, the rest as (code, count) pairs --
	 * the same table as kmer_cuda_submit_count(), half the bytes across PCIe on mostly distinct k-mers */
	if ((canonical ? kmer_cuda_submit_count_canonical(ctx, flat, off, n, k, &uniq, &n_uniq, &pairs, &n_pairs, &n_kmers)
				   : kmer_cuda_submit_count_split(ctx, flat, off, n, k, &uniq, &n_uniq, &pairs, &n_pairs, &n_kmers)) != KMER_OK)
		kmer_gpu_raise(kmer_cuda_last_error(ctx));
	d = n_uniq + n_pairs;

	/* The library's result buffers are pinned host memory owned by the context: an ereport(ERROR) between here and the
	 * releases (palloc can fail) must not leak them in a long-lived backend. */
	void *volatile r_uniq = uniq, *volatile r_pairs = pairs, *volatile r_text = NULL; /* still to be released */

	PG_TRY();
	{
		/* text of the groups with the short varlena header already in place: d * (k+1) bytes */
		codes = (uint64_t *) palloc((d ? d : 1) * sizeof(uint64_t));
		*counts = (int64_t *) palloc((d ? d : 1) * sizeof(int64_t));
		for (i = 0; i < n_uniq; i++)
		{
			codes[i] = uniq[i];
			(*counts)[i] = 1;
		}
		for (i = 0; i < n_pairs; i++)
		{
			codes[n_uniq + i] = pairs[i].code;
			(*counts)[n_uniq + i] = (int64_t) pairs[i].count;
		}
		kmer_cuda_release(ctx, r_uniq);
		r_uniq = NULL;
		kmer_cuda_release(ctx, r_pairs);
		r_pairs = NULL;
		if (kmer_cuda_submit_decode(ctx, codes, d, k, 1, &text) != KMER_OK)
			kmer_gpu_raise(kmer_cuda_last_error(ctx));
		r_text = text;

		*kmers = (struct varlena **) palloc((d ? d : 1) * sizeof(struct varlena *));
		for (i = 0; i < d; i++)
		{
			struct varlena *v = (struct varlena *) palloc((Size) k + VARHDRSZ_SHORT);

			memcpy(v, text + i * (uint64_t) (k + 1), (size_t) k + 1); /* header byte + k lower-case bases */
			(*kmers)[i] = v;
		}
	}
	PG_CATCH();
	{
		kmer_cuda_release(ctx, r_uniq);
		kmer_cuda_release(ctx, r_pairs);
		kmer_cuda_release(ctx, r_text);
		PG_RE_THROW();
	}
	PG_END_TRY();
	kmer_cuda_release(ctx, r_text);
	*n_groups = d;
}

void
kmer_gpu_count_datums(struct varlena **dnas, uint64_t n, int k, struct varlena ***kmers, int64_t **counts,
					  uint64_t *n_groups)
{
	count_datums(dnas, n, k, false, kmers, counts, n_groups);
}

/* canonical k-mers: every group's k-mer is the smaller of a k-mer and its reverse complement */
void
kmer_gpu_canonical_count_datums(struct varlena **dnas, uint64_t n, int k, struct varlena ***kmers, int64_t **counts,
								uint64_t *n_groups)
{
	count_datums(dnas, n, k, true, kmers, counts, n_groups);
}

/* counts below this are binned by the library; the (rare) groups above it come back whole and are folded in here */
#define KMER_GPU_SPECTRUM_HIST_LEN 65536

static int
cmp_u64(const void *a, const void *b)
{
	uint64_t x = *(const uint64_t *) a, y = *(const uint64_t *) b;

	return x < y ? -1 : x > y;
}

/*
 * dnas[0..n) as for kmer_gpu_count_datums.  On return (*counts)[i], (*kmers)[i] for i < *n_out are the rows of the spectrum:
 * every count that occurs, ascending, and the number of distinct k-mers with exactly that count.
 */
static void
spectrum_datums(struct varlena **dnas, uint64_t n, int k, bool canonical, int64_t **counts, int64_t **kmers, uint64_t *n_out)
{
	kmer_cuda_ctx *ctx = kmer_gpu_context();
	uint64_t *off = (uint64_t *) palloc((n + 1) * sizeof(uint64_t));
	uint64_t total = 0, i, n_tail = 0, n_kmers = 0, m = 0;
	uint64_t *hist = NULL;
	kmer_count_pair *tail = NULL;
	char *flat;

	off[0] = 0;
	for (i = 0; i < n; i++)
	{
		total += (uint64_t) VARSIZE_ANY_EXHDR(dnas[i]);
		off[i + 1] = total;
	}
	flat = (char *) palloc(total + 16);
	for (i = 0; i < n; i++)
		memcpy(flat + off[i], VARDATA_ANY(dnas[i]), (size_t) (off[i + 1] - off[i]));
	if ((canonical ? kmer_cuda_submit_count_canonical_spectrum(ctx, flat, off, n, k, KMER_GPU_SPECTRUM_HIST_LEN, &hist, &tail,
															   &n_tail, &n_kmers)
				   : kmer_cuda_submit_count_spectrum(ctx, flat, off, n, k, KMER_GPU_SPECTRUM_HIST_LEN, &hist, &tail, &n_tail,
													 &n_kmers)) != KMER_OK)
		kmer_gpu_raise(kmer_cuda_last_error(ctx));

	void *volatile r_hist = hist, *volatile r_tail = tail; /* pinned library buffers: released on every path */

	PG_TRY();
	{
		uint64_t *tc = (uint64_t *) palloc((n_tail ? n_tail : 1) * sizeof(uint64_t));
		uint64_t rows = n_tail;

		for (i = 1; i < KMER_GPU_SPECTRUM_HIST_LEN; i++)
			rows += hist[i] != 0;
		*counts = (int64_t *) palloc((rows ? rows : 1) * sizeof(int64_t));
		*kmers = (int64_t *) palloc((rows ? rows : 1) * sizeof(int64_t));
		for (i = 1; i < KMER_GPU_SPECTRUM_HIST_LEN; i++)
			if (hist[i])
			{
				(*counts)[m] = (int64_t) i;
				(*kmers)[m++] = (int64_t) hist[i];
			}
		/* the tail: one group per high-copy k-mer, every count >= KMER_GPU_SPECTRUM_HIST_LEN -- sorted and grouped by count */
		for (i = 0; i < n_tail; i++)
			tc[i] = tail[i].count;
		qsort(tc, n_tail, sizeof(uint64_t), cmp_u64);
		for (i = 0; i < n_tail; i++)
		{
			if (i && tc[i] == tc[i - 1])
				(*kmers)[m - 1]++;
			else
			{
				(*counts)[m] = (int64_t) tc[i];
				(*kmers)[m++] = 1;
			}
		}
	}
	PG_CATCH();
	{
		kmer_cuda_release(ctx, r_hist);
		kmer_cuda_release(ctx, r_tail);
		PG_RE_THROW();
	}
	PG_END_TRY();
	kmer_cuda_release(ctx, r_hist);
	kmer_cuda_release(ctx, r_tail);
	*n_out = m;
}

void
kmer_gpu_spectrum_datums(struct varlena **dnas, uint64_t n, int k, int64_t **counts, int64_t **kmers, uint64_t *n_out)
{
	spectrum_datums(dnas, n, k, false, counts, kmers, n_out);
}

void
kmer_gpu_canonical_spectrum_datums(struct varlena **dnas, uint64_t n, int k, int64_t **counts, int64_t **kmers, uint64_t *n_out)
{
	spectrum_datums(dnas, n, k, true, counts, kmers, n_out);
}

/*
 * op: KMER_OP_EQUALS (kmer = const), KMER_OP_STARTS_WITH (kmer ^@ const), KMER_OP_CONTAINS (const::qkmer @> kmer).
 * kmers[0..n) are `kmer` datums of any lengths 0..32; result[i] is the boolean the reference returns.
 */
void
kmer_gpu_match_datums(int op, struct varlena **kmers, uint64_t n, const char *constant, bool *result)
{
	kmer_cuda_ctx *ctx = kmer_gpu_context();
	char *text = (char *) palloc((n ? n : 1) * KMER_CUDA_MAX_K);
	uint8_t *lens = (uint8_t *) palloc(n ? n : 1);
	uint64_t *codes = NULL, *hits = NULL, wpr = 0, i;
	uint32_t *bits = NULL;
	const char *consts[1];

	memset(text, 'a', (n ? n : 1) * KMER_CUDA_MAX_K);
	for (i = 0; i < n; i++)
	{
		lens[i] = (uint8_t) VARSIZE_ANY_EXHDR(kmers[i]);
		memcpy(text + i * KMER_CUDA_MAX_K, VARDATA_ANY(kmers[i]), lens[i]);
	}
	if (kmer_cuda_submit_encode(ctx, text, lens, n, KMER_CUDA_MAX_K, &codes) != KMER_OK)
		kmer_gpu_raise(kmer_cuda_last_error(ctx));
	consts[0] = constant;
	if (kmer_cuda_submit_match(ctx, op, NULL, codes, lens, n, 0, consts, 1, &bits, &wpr, &hits) != KMER_OK)
	{
		kmer_cuda_release(ctx, codes);
		kmer_gpu_raise(kmer_cuda_last_error(ctx));
	}
	for (i = 0; i < n; i++)
		result[i] = (bits[i >> 5] >> (i & 31)) & 1u;
	kmer_cuda_release(ctx, codes);
	kmer_cuda_release(ctx, bits);
	kmer_cuda_release(ctx, hits);
}


/* ------------------------------------------------------------------------------------------------------------------
 * fmgr-V1 entry points (SQL-callable)
 */

typedef struct CountsState
{
	struct varlena **kmers;
	int64_t *counts;
	TupleDesc tupdesc;
} CountsState;

/*
 * kmer_gpu_counts(dna[], k) -> setof (kmer, bigint): value-per-call SRF like generate_kmers (kmer.c:289-351); the whole
 * batch is counted on the first call, in the multi-call memory context.  canonical: kmer_gpu_canonical_counts.
 */
static Datum
counts_srf(FunctionCallInfo fcinfo, bool canonical)
{
	FuncCallContext *funcctx;
	CountsState *st;

	if (SRF_IS_FIRSTCALL())
	{
		MemoryContext oldcontext;
		ArrayType *arr = PG_GETARG_ARRAYTYPE_P(0);
		int32 k = PG_GETARG_INT32(1);
		Datum *elems;
		bool *nulls;
		int n, i, m = 0;
		struct varlena **dnas;
		uint64_t n_groups = 0;
		TupleDesc tupdesc;

		funcctx = SRF_FIRSTCALL_INIT();
		oldcontext = MemoryContextSwitchTo(funcctx->multi_call_memory_ctx);
		if (get_call_result_type(fcinfo, NULL, &tupdesc) != TYPEFUNC_COMPOSITE)
			ereport(ERROR, (errcode(ERRCODE_INTERNAL_ERROR), errmsg("%s must return a composite type",
																	canonical ? "kmer_gpu_canonical_counts" : "kmer_gpu_counts")));
		deconstruct_array(arr, ARR_ELEMTYPE(arr), -1, false, 'i', &elems, &nulls, &n);
		dnas = (struct varlena **) palloc((n ? n : 1) * sizeof(struct varlena *));
		for (i = 0; i < n; i++)
			if (!nulls || !nulls[i]) /* generate_kmers is STRICT: a NULL dna yields no rows (kmer--1.0.0.sql:101-104) */
				dnas[m++] = PG_DETOAST_DATUM(elems[i]);
		st = (CountsState *) palloc(sizeof(CountsState));
		st->tupdesc = BlessTupleDesc(tupdesc);
		count_datums(dnas, (uint64_t) m, k, canonical, &st->kmers, &st->counts, &n_groups);
		funcctx->max_calls = n_groups;
		funcctx->user_fctx = st;
		MemoryContextSwitchTo(oldcontext);
	}
	funcctx = SRF_PERCALL_SETUP();
	st = (CountsState *) funcctx->user_fctx;
	if (funcctx->call_cntr < funcctx->max_calls)
	{
		Datum values[2];
		bool isnull[2] = {false, false};

		Datum tuple;

		values[0] = PointerGetDatum(st->kmers[funcctx->call_cntr]);
		values[1] = Int64GetDatum(st->counts[funcctx->call_cntr]);
		tuple = HeapTupleGetDatum(heap_form_tuple(st->tupdesc, values, isnull)); /* before SRF_RETURN_NEXT bumps call_cntr */
		SRF_RETURN_NEXT(funcctx, tuple);
	}
	SRF_RETURN_DONE(funcctx);
}

PG_FUNCTION_INFO_V1(kmer_gpu_counts);
Datum
kmer_gpu_counts(PG_FUNCTION_ARGS)
{
	return counts_srf(fcinfo, false);
}

PG_FUNCTION_INFO_V1(kmer_gpu_canonical_counts);
/* kmer_gpu_canonical_counts(dna[], k) -> setof (kmer, bigint): one row per canonical k-mer, counted over both orientations */
Datum
kmer_gpu_canonical_counts(PG_FUNCTION_ARGS)
{
	return counts_srf(fcinfo, true);
}

typedef struct SpectrumState
{
	int64_t *counts;
	int64_t *kmers;
	TupleDesc tupdesc;
} SpectrumState;

/*
 * kmer_gpu_count_spectrum(dna[], k) -> setof (count bigint, kmers bigint), ascending by count: the abundance spectrum of
 * kmer_gpu_counts(dna[], k), computed without materialising the groups.  The batch is counted on the first call.
 * canonical: kmer_gpu_canonical_count_spectrum, the spectrum of kmer_gpu_canonical_counts.
 */
static Datum
spectrum_srf(FunctionCallInfo fcinfo, bool canonical)
{
	FuncCallContext *funcctx;
	SpectrumState *st;

	if (SRF_IS_FIRSTCALL())
	{
		MemoryContext oldcontext;
		ArrayType *arr = PG_GETARG_ARRAYTYPE_P(0);
		int32 k = PG_GETARG_INT32(1);
		Datum *elems;
		bool *nulls;
		int n, i, m = 0;
		struct varlena **dnas;
		uint64_t n_rows = 0;
		TupleDesc tupdesc;

		funcctx = SRF_FIRSTCALL_INIT();
		oldcontext = MemoryContextSwitchTo(funcctx->multi_call_memory_ctx);
		if (get_call_result_type(fcinfo, NULL, &tupdesc) != TYPEFUNC_COMPOSITE)
			ereport(ERROR, (errcode(ERRCODE_INTERNAL_ERROR),
							errmsg("%s must return a composite type",
								   canonical ? "kmer_gpu_canonical_count_spectrum" : "kmer_gpu_count_spectrum")));
		deconstruct_array(arr, ARR_ELEMTYPE(arr), -1, false, 'i', &elems, &nulls, &n);
		dnas = (struct varlena **) palloc((n ? n : 1) * sizeof(struct varlena *));
		for (i = 0; i < n; i++)
			if (!nulls || !nulls[i]) /* generate_kmers is STRICT: a NULL dna yields no rows */
				dnas[m++] = PG_DETOAST_DATUM(elems[i]);
		st = (SpectrumState *) palloc(sizeof(SpectrumState));
		st->tupdesc = BlessTupleDesc(tupdesc);
		spectrum_datums(dnas, (uint64_t) m, k, canonical, &st->counts, &st->kmers, &n_rows);
		funcctx->max_calls = n_rows;
		funcctx->user_fctx = st;
		MemoryContextSwitchTo(oldcontext);
	}
	funcctx = SRF_PERCALL_SETUP();
	st = (SpectrumState *) funcctx->user_fctx;
	if (funcctx->call_cntr < funcctx->max_calls)
	{
		Datum values[2];
		bool isnull[2] = {false, false};
		Datum tuple;

		values[0] = Int64GetDatum(st->counts[funcctx->call_cntr]);
		values[1] = Int64GetDatum(st->kmers[funcctx->call_cntr]);
		tuple = HeapTupleGetDatum(heap_form_tuple(st->tupdesc, values, isnull)); /* before SRF_RETURN_NEXT bumps call_cntr */
		SRF_RETURN_NEXT(funcctx, tuple);
	}
	SRF_RETURN_DONE(funcctx);
}

PG_FUNCTION_INFO_V1(kmer_gpu_count_spectrum);
Datum
kmer_gpu_count_spectrum(PG_FUNCTION_ARGS)
{
	return spectrum_srf(fcinfo, false);
}

PG_FUNCTION_INFO_V1(kmer_gpu_canonical_count_spectrum);
Datum
kmer_gpu_canonical_count_spectrum(PG_FUNCTION_ARGS)
{
	return spectrum_srf(fcinfo, true);
}

PG_FUNCTION_INFO_V1(kmer_gpu_match);
/*
 * kmer_gpu_match(kmer[], constant text, op) -> setof boolean, element order: the batched form of kmer_equals /
 * kmer_starts_with_op / kmer_contains (kmer.c:226-285).  The constant arrives as text so that one function serves kmer and
 * qkmer constants; it is validated by the library with kmer_in's / qkmer_in's rules and messages.
 */
Datum
kmer_gpu_match(PG_FUNCTION_ARGS)
{
	FuncCallContext *funcctx;
	bool *res;

	if (SRF_IS_FIRSTCALL())
	{
		MemoryContext oldcontext;
		ArrayType *arr = PG_GETARG_ARRAYTYPE_P(0);
		struct varlena *ctext = PG_GETARG_VARLENA_P(1);
		int32 op = PG_GETARG_INT32(2);
		Datum *elems;
		bool *nulls;
		int n, i;
		struct varlena **kmers;
		char *constant;

		funcctx = SRF_FIRSTCALL_INIT();
		oldcontext = MemoryContextSwitchTo(funcctx->multi_call_memory_ctx);
		deconstruct_array(arr, ARR_ELEMTYPE(arr), -1, false, 'i', &elems, &nulls, &n);
		kmers = (struct varlena **) palloc((n ? n : 1) * sizeof(struct varlena *));
		for (i = 0; i < n; i++)
			kmers[i] = PG_DETOAST_DATUM(elems[i]);
		constant = (char *) palloc((Size) VARSIZE_ANY_EXHDR(ctext) + 1);
		memcpy(constant, VARDATA_ANY(ctext), (size_t) VARSIZE_ANY_EXHDR(ctext));
		constant[VARSIZE_ANY_EXHDR(ctext)] = 0;
		res = (bool *) palloc((n ? n : 1) * sizeof(bool));
		kmer_gpu_match_datums(op, kmers, (uint64_t) n, constant, res);
		funcctx->max_calls = (uint64_t) n;
		funcctx->user_fctx = res;
		MemoryContextSwitchTo(oldcontext);
	}
	funcctx = SRF_PERCALL_SETUP();
	res = (bool *) funcctx->user_fctx;
	if (funcctx->call_cntr < funcctx->max_calls)
	{
		/* SRF_RETURN_NEXT increments call_cntr BEFORE it evaluates its result argument: take the element first
		 * (found by executing this function against the reference, tests/c/glue_driver.c) */
		Datum d = BoolGetDatum(res[funcctx->call_cntr]);

		SRF_RETURN_NEXT(funcctx, d);
	}
	SRF_RETURN_DONE(funcctx);
}
