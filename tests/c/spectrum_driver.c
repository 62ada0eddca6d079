/* tests/c/spectrum_driver.c -- executes kmer_gpu_count_spectrum (kmer-extension_b200/pgglue/kmer_gpu.c) the way the executor
 * would: an fmgr-V1 call through the pgshim, `dna` varlenas of both header forms, value-per-call SRF protocol.  The expected
 * side is the spectrum of the GROUP BY the reference's generate_kmers produces (tests/c/expected_kmers.h: the reference's own
 * function, or the C oracle with -DPGSHIM_NO_REFERENCE):
 *   SELECT cnt, count(*) FROM (SELECT count(*) AS cnt FROM reads r, generate_kmers(r.dna, k) g GROUP BY g.kmer) s
 *   GROUP BY cnt ORDER BY cnt
 * Rows must be equal in number, order and value; errors must carry the reference's SQLSTATE and text.  Built and run by
 * tests/test_spectrum_glue.py.  Exit code 0 = all equal. */
#include "postgres.h"
#include "fmgr.h"
#include "funcapi.h"
#include "utils/array.h"

extern Datum kmer_gpu_count_spectrum(PG_FUNCTION_ARGS);

static uint64_t rng_state = 0x2545F4914F6CDD1DULL;
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

/* n_rows random reads of k..max_len bases; every repeat_every-th read is the same one (counts above 1); n_homo reads of
 * homo_len identical bases (one k-mer counted homo_len-k+1 times: beyond the library's histogram at homo_len > 65556) */
static int check_spectrum(int n_rows, int max_len, int k, int repeat_every, int n_homo, int homo_len)
{
	int total_rows = n_rows + n_homo;
	ArrayType *arr = (ArrayType *) palloc(sizeof(ArrayType) + (size_t) total_rows * sizeof(Datum));
	Item *want = NULL;
	size_t n_want = 0, cap_want = 0;
	int buf_len = max_len > homo_len ? max_len : homo_len;
	char *buf = (char *) palloc((Size) buf_len + 1);
	arr->nelems = total_rows;
	arr->elemtype = 0;
	for (int r = 0; r < total_rows; r++)
	{
		int len;
		if (r < n_rows)
		{
			len = k + (int) (rnd() % (uint32_t) (max_len - k + 1));
			if (repeat_every && r % repeat_every == 0) rng_state = 7;
			for (int i = 0; i < len; i++) buf[i] = "ACGTacgt"[rnd() & 7];
		}
		else
		{
			len = homo_len;
			memset(buf, "AcGt"[(r - n_rows) & 3], (size_t) len);
		}
		arr->elems[r] = PointerGetDatum(make_varlena(buf, len, r & 1));
		char *low = (char *) palloc((Size) len);
		for (int i = 0; i < len; i++) low[i] = (char) (buf[i] | 0x20);
		want = expected_kmers(want, &n_want, &cap_want, low, len, k);
	}
	/* the expected side: GROUP BY kmer, then GROUP BY count */
	qsort(want, n_want, sizeof(Item), cmp_item);
	int64_t *cnt = (int64_t *) malloc((n_want + 1) * sizeof(int64_t));
	size_t g = 0;
	for (size_t i = 0; i < n_want; i++)
	{
		if (i && !memcmp(want[i - 1].bytes, want[i].bytes, 40)) cnt[g - 1]++;
		else cnt[g++] = 1;
	}
	qsort(cnt, g, sizeof(int64_t), cmp_i64);
	int64_t *wc = (int64_t *) malloc((g + 1) * sizeof(int64_t)), *wk = (int64_t *) malloc((g + 1) * sizeof(int64_t));
	size_t nw = 0;
	for (size_t i = 0; i < g; i++)
	{
		if (nw && wc[nw - 1] == cnt[i]) wk[nw - 1]++;
		else { wc[nw] = cnt[i]; wk[nw++] = 1; }
	}
	/* the glue */
	FunctionCallInfoBaseData fc;
	memset(&fc, 0, sizeof(fc));
	fc.nargs = 2;
	fc.args[0].value = PointerGetDatum(arr);
	fc.args[1].value = (Datum) k;
	size_t n_got = 0;
	int ok = 1;
	for (;;)
	{
		Datum d = kmer_gpu_count_spectrum(&fc);
		if (fc.srf_done) break;
		HeapTuple t = (HeapTuple) DatumGetPointer(d);
		int64_t c = DatumGetInt64(t->values[0]), m = DatumGetInt64(t->values[1]);
		if (n_got >= nw || c != wc[n_got] || m != wk[n_got])
		{
			if (ok) printf("       first mismatch at row %zu: glue (%lld, %lld)\n", n_got, (long long) c, (long long) m);
			ok = 0;
		}
		n_got++;
	}
	ok = ok && n_got == nw;
	printf("[glue] kmer_gpu_count_spectrum: %d rows (both header forms), k=%d: %s  spectrum rows %zu/%zu, groups %zu, k-mers %zu, "
		   "largest count %lld (expected side: %s)\n", total_rows, k, ok ? "ok" : "MISMATCH", n_got, nw, g, n_want,
		   nw ? (long long) wc[nw - 1] : 0LL, EXPECTED_SOURCE);
	free(want); free(cnt); free(wc); free(wk);
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
		kmer_gpu_count_spectrum(&fc);
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
	ok &= check_spectrum(3000, 120, 21, 0, 0, 0);
	ok &= check_spectrum(2000, 90, 31, 5, 0, 0);
	ok &= check_spectrum(4000, 60, 5, 0, 0, 0);
	ok &= check_spectrum(1500, 100, 32, 7, 0, 0);
	ok &= check_spectrum(1, 21, 21, 0, 0, 0);
	ok &= check_spectrum(500, 80, 21, 3, 3, 70000);   /* three tail groups with one count */
	ok &= check_spectrum(300, 80, 32, 0, 4, 66000);   /* k = 32: poly-T is the all-ones code */
	ok &= check_error("ACGTNACGTACGTACGTACGTACGTACGT", 21, ERRCODE_INVALID_TEXT_REPRESENTATION, "Invalid DNA Sequence");
	ok &= check_error("ACGT", 21, ERRCODE_INVALID_PARAMETER_VALUE, "Invalid KMER Length");
	ok &= check_error("ACGTACGTACGTACGTACGTACGT", 33, ERRCODE_INVALID_PARAMETER_VALUE, "Invalid KMER Length");
	return ok ? 0 : 1;
}
