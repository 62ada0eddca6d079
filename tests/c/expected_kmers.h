/* tests/c/expected_kmers.h -- the expected side of tests/c/glue_driver.c and tests/c/hook_driver.c: the k-mer datums
 * generate_kmers(dna, k) returns for one row, and the predicates on one k-mer.  Linked with the reference (oracle/_ref) they
 * come from the reference's own functions.  Built with -DPGSHIM_NO_REFERENCE they come from the C oracle
 * (oracle/kmer_oracle.c, libkmer_oracle.so), which tests/test_oracle.py pins to the answers the reference recorded
 * (tests/golden).  Include after make_varlena(). */
#ifndef EXPECTED_KMERS_H
#define EXPECTED_KMERS_H

typedef struct Item { unsigned char bytes[40]; int64_t count; } Item; /* a kmer datum: header byte + <= 32 bases */
static int cmp_item(const void *a, const void *b) { return memcmp(((const Item *) a)->bytes, ((const Item *) b)->bytes, 40); }

static Item *push_item(Item *v, size_t *n, size_t *cap)
{
	if (*n == *cap)
	{
		*cap = *cap ? *cap * 2 : 4096;
		v = (Item *) realloc(v, *cap * sizeof(Item));
	}
	memset(&v[*n], 0, sizeof(Item));
	v[*n].count = 1;
	(*n)++;
	return v;
}

#ifdef PGSHIM_NO_REFERENCE
#define EXPECTED_SOURCE "the C oracle"
extern int orc_generate(const char *flat, const uint64_t *off, uint64_t n_rows, int k, uint64_t *codes, uint64_t *n_out, int64_t *bad_row);
extern void orc_kmer_decode(uint64_t code, int k, char *out);
extern int orc_kmer_encode(const char *s, uint64_t len, uint64_t *code);
extern int orc_match_column(int op, const uint64_t *codes, const uint8_t *lens, uint64_t m, int k, const char *const_text, uint8_t *out);

/* generate_kmers over one row (lower-case bases, as dna_in stores them): one datum per window, in position order */
static Item *expected_kmers(Item *want, size_t *n, size_t *cap, const char *low, int len, int k)
{
	uint64_t off[2] = {0, (uint64_t) len}, m = 0;
	int64_t bad;
	uint64_t *codes = (uint64_t *) malloc(((size_t) len + 1) * sizeof(uint64_t));
	if (orc_generate(low, off, 1, k, codes, &m, &bad)) { printf("oracle: generate_kmers rejects a row\n"); exit(2); }
	for (uint64_t i = 0; i < m; i++)
	{
		want = push_item(want, n, cap);
		SET_VARSIZE_SHORT(want[*n - 1].bytes, k + 1);            /* the datum's 1-byte header (kmer.c:341-343) */
		orc_kmer_decode(codes[i], k, (char *) want[*n - 1].bytes + 1);
	}
	free(codes);
	return want;
}

/* op 0: kmer = constant, 1: kmer ^@ constant, 2: constant::qkmer @> kmer -- on a k-mer of len lower-case bases */
static int expected_match(int op, const char *kmer, int len, const char *constant)
{
	uint64_t code = 0;
	uint8_t l = (uint8_t) len, r = 0;
	if (orc_kmer_encode(kmer, (uint64_t) len, &code) || orc_match_column(op, &code, &l, 1, len, constant, &r))
	{
		printf("oracle: rejects k-mer '%.*s' or constant '%s'\n", len, kmer, constant);
		exit(2);
	}
	return r;
}
#else
#define EXPECTED_SOURCE "the reference"
extern Datum generate_kmers(PG_FUNCTION_ARGS);

/* one generate_kmers SRF scan of one row: the datums exactly as the reference palloc's them */
static Item *expected_kmers(Item *want, size_t *n, size_t *cap, const char *low, int len, int k)
{
	FunctionCallInfoBaseData fc;
	memset(&fc, 0, sizeof(fc));
	fc.nargs = 2;
	fc.args[0].value = PointerGetDatum(make_varlena(low, len, 0));
	fc.args[1].value = (Datum) k;
	for (;;)
	{
		Datum d = generate_kmers(&fc);
		if (fc.srf_done) break;
		want = push_item(want, n, cap);
		memcpy(want[*n - 1].bytes, DatumGetPointer(d), (size_t) k + 1);
	}
	return want;
}
#endif

#endif /* EXPECTED_KMERS_H */
