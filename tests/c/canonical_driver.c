/* tests/c/canonical_driver.c -- executes kmer_gpu_canonical_counts and kmer_gpu_canonical_count_spectrum
 * (kmer-extension_b200/pgglue/kmer_gpu.c) the way the executor would: fmgr-V1 calls through the pgshim, `dna` varlenas of both
 * header forms, value-per-call SRF protocol.  The expected side folds the k-mer datums the reference's generate_kmers
 * produces (tests/c/expected_kmers.h: the reference's own function, or the C oracle with -DPGSHIM_NO_REFERENCE) canonically:
 *   SELECT least(g.kmer::text COLLATE "C", reverse(translate(g.kmer::text, 'acgt', 'tgca')))::kmer, count(*)
 *   FROM reads r, generate_kmers(r.dna, k) g GROUP BY 1
 * and the spectrum of that table.  Groups must be equal as a set, spectrum rows in number, order and value; errors must carry
 * the reference's SQLSTATE and text.  Built and run by tests/test_canonical_glue.py.  Exit code 0 = all equal. */
#include "postgres.h"
#include "fmgr.h"
#include "funcapi.h"
#include "utils/array.h"

extern Datum kmer_gpu_canonical_counts(PG_FUNCTION_ARGS);
extern Datum kmer_gpu_canonical_count_spectrum(PG_FUNCTION_ARGS);

static uint64_t rng_state = 0x9E3779B97F4A7C15ULL;
static uint32_t rnd(void)
{
	rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17;
	return (uint32_t) (rng_state >> 32);
}

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

static int cmp_i64(const void *a, const void *b)
{
	int64_t x = *(const int64_t *) a, y = *(const int64_t *) b;
	return x < y ? -1 : x > y;
}

/* the k-mer text of a datum (header byte + k lower-case bases) -> the smaller of it and its reverse complement */
static void canonicalize(Item *it, int k)
{
	char rc[32];
	for (int i = 0; i < k; i++)
	{
		char b = (char) it->bytes[k - i];
		rc[i] = b == 'a' ? 't' : b == 'c' ? 'g' : b == 'g' ? 'c' : 'a';
	}
	if (memcmp(rc, it->bytes + 1, (size_t) k) < 0) memcpy(it->bytes + 1, rc, (size_t) k);
}

static ArrayType *make_rows(int n_rows, int max_len, int k, int repeat_every, int n_homo, int homo_len, Item **want, size_t *n_want)
{
	int total_rows = n_rows + n_homo;
	ArrayType *arr = (ArrayType *) palloc(sizeof(ArrayType) + (size_t) total_rows * sizeof(Datum));
	size_t cap_want = 0;
	int buf_len = (max_len > homo_len ? max_len : homo_len) * 2;
	char *buf = (char *) palloc((Size) buf_len + 1), *prev = (char *) palloc((Size) buf_len + 1);
	int prev_len = 0;
	arr->nelems = total_rows;
	arr->elemtype = 0;
	*want = NULL;
	*n_want = 0;
	for (int r = 0; r < total_rows; r++)
	{
		int len;
		if (r < n_rows && repeat_every && r % repeat_every == 1 && prev_len)
		{                                               /* the reverse complement of the previous row, case swapped */
			len = prev_len;
			for (int i = 0; i < len; i++)
			{
				char b = (char) (prev[len - 1 - i] | 0x20);
				char c = b == 'a' ? 't' : b == 'c' ? 'g' : b == 'g' ? 'c' : 'a';
				buf[i] = (prev[len - 1 - i] & 0x20) ? (char) (c & ~0x20) : c;
			}
		}
		else if (r < n_rows)
		{
			len = k + (int) (rnd() % (uint32_t) (max_len - k + 1));
			for (int i = 0; i < len; i++) buf[i] = "ACGTacgt"[rnd() & 7];
		}
		else
		{
			len = homo_len;
			memset(buf, "AcGt"[(r - n_rows) & 3], (size_t) len);
		}
		memcpy(prev, buf, (size_t) len);
		prev_len = len;
		arr->elems[r] = PointerGetDatum(make_varlena(buf, len, r & 1));
		char *low = (char *) palloc((Size) len);
		for (int i = 0; i < len; i++) low[i] = (char) (buf[i] | 0x20);
		size_t before = *n_want;
		*want = expected_kmers(*want, n_want, &cap_want, low, len, k);
		for (size_t i = before; i < *n_want; i++) canonicalize(&(*want)[i], k);
	}
	return arr;
}

static void call_args(FunctionCallInfoBaseData *fc, ArrayType *arr, int k)
{
	memset(fc, 0, sizeof(*fc));
	fc->nargs = 2;
	fc->args[0].value = PointerGetDatum(arr);
	fc->args[1].value = (Datum) k;
}

static int check(int n_rows, int max_len, int k, int repeat_every, int n_homo, int homo_len)
{
	Item *want;
	size_t n_want;
	ArrayType *arr = make_rows(n_rows, max_len, k, repeat_every, n_homo, homo_len, &want, &n_want);
	/* the expected side: GROUP BY the canonical k-mer */
	qsort(want, n_want, sizeof(Item), cmp_item);
	size_t g = 0;
	for (size_t i = 0; i < n_want; i++)
	{
		if (g && !memcmp(want[g - 1].bytes, want[i].bytes, 40)) want[g - 1].count++;
		else { want[g] = want[i]; want[g].count = 1; g++; }
	}
	/* kmer_gpu_canonical_counts */
	FunctionCallInfoBaseData fc;
	call_args(&fc, arr, k);
	Item *got = (Item *) malloc((g + 1) * sizeof(Item));
	size_t n_got = 0;
	int ok = 1;
	for (;;)
	{
		Datum d = kmer_gpu_canonical_counts(&fc);
		if (fc.srf_done) break;
		HeapTuple t = (HeapTuple) DatumGetPointer(d);
		if (n_got == g) { ok = 0; n_got++; continue; }
		memset(&got[n_got], 0, sizeof(Item));
		memcpy(got[n_got].bytes, DatumGetPointer(t->values[0]), (size_t) k + 1);
		got[n_got++].count = DatumGetInt64(t->values[1]);
	}
	ok = ok && n_got == g;
	if (ok)
	{
		qsort(got, n_got, sizeof(Item), cmp_item);
		for (size_t i = 0; i < g && ok; i++)
			if (memcmp(got[i].bytes, want[i].bytes, 40) || got[i].count != want[i].count)
			{
				printf("       first mismatch at group %zu: '%.*s' %lld, want '%.*s' %lld\n", i, k, got[i].bytes + 1,
					   (long long) got[i].count, k, want[i].bytes + 1, (long long) want[i].count);
				ok = 0;
			}
	}
	printf("[glue] kmer_gpu_canonical_counts: %d rows, k=%d: %s  groups %zu/%zu, k-mers %zu (expected side: %s)\n",
		   n_rows + n_homo, k, ok ? "ok" : "MISMATCH", n_got, g, n_want, EXPECTED_SOURCE);
	/* kmer_gpu_canonical_count_spectrum against the spectrum of the expected table */
	int64_t *cnt = (int64_t *) malloc((g + 1) * sizeof(int64_t)), *wc = (int64_t *) malloc((g + 1) * sizeof(int64_t)),
			*wk = (int64_t *) malloc((g + 1) * sizeof(int64_t));
	for (size_t i = 0; i < g; i++) cnt[i] = want[i].count;
	qsort(cnt, g, sizeof(int64_t), cmp_i64);
	size_t nw = 0, n_spec = 0;
	for (size_t i = 0; i < g; i++)
	{
		if (nw && wc[nw - 1] == cnt[i]) wk[nw - 1]++;
		else { wc[nw] = cnt[i]; wk[nw++] = 1; }
	}
	int ok2 = 1;
	call_args(&fc, arr, k);
	for (;;)
	{
		Datum d = kmer_gpu_canonical_count_spectrum(&fc);
		if (fc.srf_done) break;
		HeapTuple t = (HeapTuple) DatumGetPointer(d);
		int64_t c = DatumGetInt64(t->values[0]), m = DatumGetInt64(t->values[1]);
		if (n_spec >= nw || c != wc[n_spec] || m != wk[n_spec]) ok2 = 0;
		n_spec++;
	}
	ok2 = ok2 && n_spec == nw;
	printf("[glue] kmer_gpu_canonical_count_spectrum: k=%d: %s  spectrum rows %zu/%zu, largest count %lld\n", k,
		   ok2 ? "ok" : "MISMATCH", n_spec, nw, nw ? (long long) wc[nw - 1] : 0LL);
	free(want); free(got); free(cnt); free(wc); free(wk);
	return ok && ok2;
}

static int check_error(Datum (*fn)(PG_FUNCTION_ARGS), const char *row, int k, int sqlstate, const char *message)
{
	ArrayType *arr = (ArrayType *) palloc(sizeof(ArrayType) + 2 * sizeof(Datum));
	FunctionCallInfoBaseData fc;
	jmp_buf jb;
	int ok = 0;
	arr->nelems = 2;
	arr->elemtype = 0;
	arr->elems[0] = PointerGetDatum(make_varlena("ACGTACGTACGTACGTACGTACGTACGTACGTACGT", 36, 0));
	arr->elems[1] = PointerGetDatum(make_varlena(row, (int) strlen(row), 0));
	call_args(&fc, arr, k);
	pgshim_handler = &jb;
	if (setjmp(jb) == 0)
	{
		fn(&fc);
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
	ok &= check(3000, 120, 21, 2, 0, 0);       /* every other row is the reverse complement of the one before */
	ok &= check(2000, 90, 31, 3, 0, 0);
	ok &= check(4000, 60, 5, 0, 0, 0);
	ok &= check(1500, 100, 32, 2, 4, 200);     /* k = 32: poly-A and poly-T are one group */
	ok &= check(1, 4, 4, 0, 0, 0);
	ok &= check(500, 80, 14, 2, 3, 70000);     /* counts beyond the library's histogram */
	Datum (*fns[2])(PG_FUNCTION_ARGS) = {kmer_gpu_canonical_counts, kmer_gpu_canonical_count_spectrum};
	for (int f = 0; f < 2; f++)
	{
		ok &= check_error(fns[f], "ACGTNACGTACGTACGTACGTACGTACGT", 21, ERRCODE_INVALID_TEXT_REPRESENTATION, "Invalid DNA Sequence");
		ok &= check_error(fns[f], "ACGT", 21, ERRCODE_INVALID_PARAMETER_VALUE, "Invalid KMER Length");
		ok &= check_error(fns[f], "ACGTACGTACGTACGTACGTACGT", 33, ERRCODE_INVALID_PARAMETER_VALUE, "Invalid KMER Length");
	}
	return ok ? 0 : 1;
}
