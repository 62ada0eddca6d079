/* tests/c/glue_driver.c -- executes the PostgreSQL-side glue (kmer-extension_b200/pgglue/kmer_gpu.c) the way the executor
 * would: fmgr-V1 calls through the pgshim, `dna` / `kmer` varlenas with BOTH header forms, value-per-call SRF protocol.
 * The reference's own functions (generate_kmers, kmer_equals, kmer_starts_with_op, kmer_contains -- compiled unmodified into
 * oracle/_ref/libkmer_ref.so, which also provides the shim's palloc / ereport runtime) run in the same process on the same
 * datums; the glue's datums must equal theirs BYTE FOR BYTE (header byte included, kmer.c:341-343), its counts must equal
 * the number of times the reference emitted each k-mer, its booleans the reference's booleans, its errors the reference's
 * SQLSTATE and text.  Built with -DPGSHIM_NO_REFERENCE (no oracle/_ref) the expected side is the C oracle instead
 * (tests/c/expected_kmers.h).  Built and run by tests/test_glue_exec.py.  Exit code 0 = all equal. */
#include "postgres.h"
#include "fmgr.h"
#include "funcapi.h"
#include "utils/array.h"

extern Datum kmer_equals(PG_FUNCTION_ARGS);
extern Datum kmer_starts_with_op(PG_FUNCTION_ARGS);
extern Datum kmer_contains(PG_FUNCTION_ARGS);
extern Datum kmer_in(PG_FUNCTION_ARGS);
extern Datum qkmer_in(PG_FUNCTION_ARGS);
extern Datum kmer_gpu_counts(PG_FUNCTION_ARGS);
extern Datum kmer_gpu_match(PG_FUNCTION_ARGS);

static uint64_t rng_state = 0x9E3779B97F4A7C15ULL;
static uint32_t rnd(void)
{
	rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17;
	return (uint32_t) (rng_state >> 32);
}

/* a varlena with the 4-byte header (what dna_in builds, kmer.c:92-93) or the 1-byte short header PostgreSQL stores on disk */
static struct varlena *make_varlena(const char *bytes, int len, int short_header)
{
	struct varlena *v;
	if (short_header && len + 1 <= 127)
	{
		v = (struct varlena *) palloc((Size) len + 1);
		SET_VARSIZE_SHORT(v, len + 1);
		memcpy((char *) v + 1, bytes, (size_t) len);
	}
	else
	{
		v = (struct varlena *) palloc((Size) len + VARHDRSZ);
		SET_VARSIZE(v, len + VARHDRSZ);
		memcpy((char *) v + VARHDRSZ, bytes, (size_t) len);
	}
	return v;
}

#include "expected_kmers.h"

static int check_counts(int n_rows, int max_len, int k, int repeat_every)
{
	ArrayType *arr = (ArrayType *) palloc(sizeof(ArrayType) + (size_t) n_rows * sizeof(Datum));
	Item *want = NULL;
	size_t n_want = 0, cap_want = 0;
	char *buf = (char *) palloc((Size) max_len + 1);
	arr->nelems = n_rows;
	arr->elemtype = 0;
	for (int r = 0; r < n_rows; r++)
	{
		int len = k + (int) (rnd() % (uint32_t) (max_len - k + 1));
		if (repeat_every && r % repeat_every == 0) rng_state = 42; /* the same read again: counts above 1 */
		for (int i = 0; i < len; i++) buf[i] = "ACGTacgt"[rnd() & 7];
		arr->elems[r] = PointerGetDatum(make_varlena(buf, len, r & 1));
		/* the expected side: one generate_kmers scan of this row; dna_in lower-cases (kmer.c:28-29): hand it the stored form */
		char *low = (char *) palloc((Size) len);
		for (int i = 0; i < len; i++) low[i] = (char) (buf[i] | 0x20);
		want = expected_kmers(want, &n_want, &cap_want, low, len, k);
	}
	qsort(want, n_want, sizeof(Item), cmp_item);
	size_t g = 0;
	for (size_t i = 0; i < n_want; i++)
	{
		if (g && !memcmp(want[g - 1].bytes, want[i].bytes, 40)) want[g - 1].count++;
		else want[g++] = want[i];
	}
	/* the glue: kmer_gpu_counts(dna[], k) until done */
	FunctionCallInfoBaseData fc;
	memset(&fc, 0, sizeof(fc));
	fc.nargs = 2;
	fc.args[0].value = PointerGetDatum(arr);
	fc.args[1].value = (Datum) k;
	Item *got = (Item *) malloc((g + 16) * sizeof(Item));
	size_t n_got = 0;
	for (;;)
	{
		Datum d = kmer_gpu_counts(&fc);
		if (fc.srf_done) break;
		HeapTuple t = (HeapTuple) DatumGetPointer(d);
		if (n_got < g + 16)
		{
			struct varlena *v = (struct varlena *) DatumGetPointer(t->values[0]);
			memset(&got[n_got], 0, sizeof(Item));
			memcpy(got[n_got].bytes, v, (size_t) VARSIZE_SHORT(v));
			got[n_got].count = DatumGetInt64(t->values[1]);
		}
		n_got++;
	}
	qsort(got, n_got < g + 16 ? n_got : g + 16, sizeof(Item), cmp_item);
	int ok = n_got == g;
	for (size_t i = 0; ok && i < g; i++) ok = !memcmp(got[i].bytes, want[i].bytes, 40) && got[i].count == want[i].count;
	printf("[glue] kmer_gpu_counts: %d rows (both header forms), k=%d: %s  groups %zu/%zu, k-mers %zu (expected side: %s)\n", n_rows, k,
		   ok ? "ok" : "MISMATCH", n_got, g, n_want, EXPECTED_SOURCE);
	free(want); free(got);
	return ok;
}

static int check_match(int n, int op, const char *constant)
{
	ArrayType *arr = (ArrayType *) palloc(sizeof(ArrayType) + (size_t) n * sizeof(Datum));
	int ok = 1, hits = 0;
	FunctionCallInfoBaseData fc;
	arr->nelems = n;
	arr->elemtype = 0;
#ifndef PGSHIM_NO_REFERENCE
	/* the constant through the reference's own input function */
	memset(&fc, 0, sizeof(fc));
	fc.nargs = 1;
	fc.args[0].value = PointerGetDatum(pstrdup(constant));
	Datum cst = op == 2 ? qkmer_in(&fc) : kmer_in(&fc);
#endif
	unsigned char *want = (unsigned char *) palloc((Size) n);
	int clen = (int) strlen(constant);
	for (int i = 0; i < n; i++)
	{
		char b[33];
		int len = (i % 7 == 0) ? clen : (int) (rnd() % 33);
		for (int j = 0; j < len; j++) b[j] = "acgt"[rnd() & 3];
		if (i % 3 == 0) /* make hits likely: copy the constant's definite letters */
			for (int j = 0; j < len && j < clen; j++)
				if (strchr("acgtACGT", constant[j])) b[j] = (char) (constant[j] | 0x20);
		struct varlena *v = make_varlena(b, len, 1); /* kmer datums carry the short header (kmer.c:124-125) */
		arr->elems[i] = PointerGetDatum(v);
#ifdef PGSHIM_NO_REFERENCE
		want[i] = (unsigned char) expected_match(op, b, len, constant);
#else
		memset(&fc, 0, sizeof(fc));
		fc.nargs = 2;
		if (op == 0) { fc.args[0].value = PointerGetDatum(v); fc.args[1].value = cst; want[i] = kmer_equals(&fc) != 0; }
		else if (op == 1) { fc.args[0].value = PointerGetDatum(v); fc.args[1].value = cst; want[i] = kmer_starts_with_op(&fc) != 0; }
		else { fc.args[0].value = cst; fc.args[1].value = PointerGetDatum(v); want[i] = kmer_contains(&fc) != 0; }
#endif
		hits += want[i];
	}
	memset(&fc, 0, sizeof(fc));
	fc.nargs = 3;
	fc.args[0].value = PointerGetDatum(arr);
	fc.args[1].value = PointerGetDatum(make_varlena(constant, clen, 0));
	fc.args[2].value = (Datum) op;
	int i = 0, got_hits = 0, first_bad = -1;
	for (;; i++)
	{
		Datum d = kmer_gpu_match(&fc);
		if (fc.srf_done) break;
		got_hits += DatumGetBool(d);
		if (i < n && DatumGetBool(d) != (want[i] != 0)) { ok = 0; if (first_bad < 0) first_bad = i; }
	}
	ok = ok && i == n;
	printf("[glue] kmer_gpu_match op=%d const=%s: %d kmers, %d hits (glue %d, %d results): %s\n", op, constant, n, hits, got_hits, i,
		   ok ? "ok" : "MISMATCH");
	if (first_bad >= 0)
	{
		struct varlena *v = (struct varlena *) DatumGetPointer(arr->elems[first_bad]);
		printf("       first mismatch at element %d: kmer '%.*s' (len %d), " EXPECTED_SOURCE " says %d\n", first_bad, (int) VARSIZE_ANY_EXHDR(v), VARDATA_ANY(v),
			   (int) VARSIZE_ANY_EXHDR(v), (int) want[first_bad]);
	}
	return ok;
}

static int check_error(const char *row, int k, int sqlstate, const char *message)
{
	ArrayType *arr = (ArrayType *) palloc(sizeof(ArrayType) + 2 * sizeof(Datum));
	FunctionCallInfoBaseData fc;
	jmp_buf jb;
	int ok = 0;
	arr->nelems = 2;
	arr->elemtype = 0;
	arr->elems[0] = PointerGetDatum(make_varlena("ACGTACGTACGTACGTACGTACGTACGTACGTACGT", 36, 0));
	arr->elems[1] = PointerGetDatum(make_varlena(row, (int) strlen(row), 0));
	memset(&fc, 0, sizeof(fc));
	fc.nargs = 2;
	fc.args[0].value = PointerGetDatum(arr);
	fc.args[1].value = (Datum) k;
	pgshim_handler = &jb;
	if (setjmp(jb) == 0)
	{
		kmer_gpu_counts(&fc);
		printf("[glue] expected ERROR %s, got a result\n", message);
	}
	else
		ok = pgshim_error.sqlstate == sqlstate && !strcmp(pgshim_error.message, message);
	pgshim_handler = NULL;
	printf("[glue] ereport: \"%s\" sqlstate %x: %s\n", pgshim_error.message, pgshim_error.sqlstate, ok ? "ok" : "MISMATCH");
	return ok;
}

int main(void)
{
	int ok = 1;
	ok &= check_counts(3000, 120, 21, 0);
	ok &= check_counts(2000, 90, 31, 5);
	ok &= check_counts(4000, 60, 5, 0);
	ok &= check_counts(1500, 100, 32, 7);
	ok &= check_counts(1, 21, 21, 0);
	ok &= check_match(5000, 0, "acgtacgt");
	ok &= check_match(5000, 1, "ACG");
	ok &= check_match(5000, 2, "ANGRYacg");
	ok &= check_match(5000, 2, "");
	ok &= check_error("ACGTNACGTACGTACGTACGTACGTACGT", 21, ERRCODE_INVALID_TEXT_REPRESENTATION, "Invalid DNA Sequence");
	ok &= check_error("ACGT", 21, ERRCODE_INVALID_PARAMETER_VALUE, "Invalid KMER Length");
	return ok ? 0 : 1;
}
