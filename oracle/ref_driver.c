/*
 * oracle/ref_driver.c -- TEST INFRASTRUCTURE ONLY (never linked into libkmer_cuda.so).
 *
 * Executor stand-in around the UNMODIFIED reference extension source.  The Makefile in this
 * directory compiles /root/reference/kmer.c in place (it is never copied into this repository)
 * together with this file into oracle/_ref/libkmer_ref.so.  Everything the reference computes
 * is computed by the reference's own functions, called through their fmgr-V1 entry points:
 *
 *   dna_in / kmer_in / qkmer_in      kmer.c:84-97, 109-129, 141-190
 *   generate_kmers (SRF)             kmer.c:289-351
 *   kmer_hash / kmer_equals          kmer.c:353-365, 226-245   (GROUP BY support)
 *   kmer_starts_with / _op           kmer.c:248-265
 *   kmer_contains / kmer_containing  kmer.c:268-285
 *
 * What this file adds is only what PostgreSQL core supplies in a real server: palloc, ereport,
 * the value-per-call SRF loop (ExecMakeTableFunctionResult), and a HashAggregate + count(*)
 * (nodeAgg.c) keyed through the extension's hash opclass, i.e. hash(kmer) for the bucket and
 * equals(kmer,kmer) on every hash hit -- with Partial/Finalize aggregation over worker threads
 * shaped like a parallel plan (Gather over Partial HashAggregate).
 */
#include "postgres.h"
#include "fmgr.h"
#include "funcapi.h"
#include "access/hash.h"
#include <pthread.h>

int pgshim_module_magic = 1;

/* ------------------------------------------------------------------ memory */

typedef struct ArenaBlock
{
	struct ArenaBlock *next;
	size_t cap, used;
	char data[];
} ArenaBlock;

typedef struct PgShimArena
{
	ArenaBlock *head;
} PgShimArena;

static __thread PgShimArena tl_arena;

static void *arena_alloc(PgShimArena *a, size_t n)
{
	n = (n + 15) & ~(size_t) 15;
	if (!a->head || a->head->used + n > a->head->cap)
	{
		size_t cap = n > (1u << 16) ? n : (1u << 16);
		ArenaBlock *b = (ArenaBlock *) malloc(sizeof(ArenaBlock) + cap);
		if (!b)
			abort();
		b->cap = cap;
		b->used = 0;
		b->next = a->head;
		a->head = b;
	}
	void *p = a->head->data + a->head->used;
	a->head->used += n;
	return p;
}

/* per-row reset: keep one block, like resetting a per-tuple memory context */
static void arena_reset(PgShimArena *a)
{
	while (a->head && a->head->next)
	{
		ArenaBlock *n = a->head->next;
		free(a->head);
		a->head = n;
	}
	if (a->head)
		a->head->used = 0;
}

static void arena_free(PgShimArena *a)
{
	while (a->head)
	{
		ArenaBlock *n = a->head->next;
		free(a->head);
		a->head = n;
	}
}

void *pgshim_palloc(Size n) { return arena_alloc(&tl_arena, n ? n : 1); }

char *pgshim_pstrdup(const char *s)
{
	size_t n = strlen(s) + 1;
	char *p = (char *) pgshim_palloc(n);
	memcpy(p, s, n);
	return p;
}

char *pgshim_psprintf(const char *fmt, ...)
{
	va_list ap, ap2;
	va_start(ap, fmt);
	va_copy(ap2, ap);
	int n = vsnprintf(NULL, 0, fmt, ap);
	va_end(ap);
	char *p = (char *) pgshim_palloc((size_t) n + 1);
	vsnprintf(p, (size_t) n + 1, fmt, ap2);
	va_end(ap2);
	return p;
}

void pgshim_pfree(void *p) { (void) p; } /* bump arena: freed by the reset */

/* composite results for the GPU glue's SRFs (funcapi.h) */
TypeFuncClass pgshim_get_call_result_type(FunctionCallInfo fcinfo, Oid *resultTypeId, TupleDesc *resultTupleDesc)
{
	(void) fcinfo;
	if (resultTypeId)
		*resultTypeId = 0;
	TupleDesc d = (TupleDesc) pgshim_palloc(sizeof(*d));
	d->natts = 2;
	*resultTupleDesc = d;
	return TYPEFUNC_COMPOSITE;
}

HeapTuple pgshim_heap_form_tuple(TupleDesc desc, Datum *values, bool *isnull)
{
	HeapTuple t = (HeapTuple) pgshim_palloc(sizeof(*t));
	t->natts = desc->natts;
	for (int i = 0; i < desc->natts && i < 8; i++)
	{
		t->values[i] = values[i];
		t->nulls[i] = isnull ? isnull[i] : false;
	}
	return t;
}

/* exported for test drivers outside this file (tests/c/glue_driver.c): per-statement reset of the palloc arena */
void pgshim_reset(void);

FuncCallContext *pgshim_srf_firstcall_init(FunctionCallInfo fcinfo)
{
	FuncCallContext *c = (FuncCallContext *) pgshim_palloc(sizeof(FuncCallContext));
	memset(c, 0, sizeof(*c));
	c->multi_call_memory_ctx = &tl_arena;
	fcinfo->srf_ctx = c;
	return c;
}

void pgshim_reset(void) { arena_reset(&tl_arena); }

/* ------------------------------------------------------------------ errors */

__thread PgShimError pgshim_error;
__thread jmp_buf *pgshim_handler;

int pgshim_errcode(int code)
{
	pgshim_error.sqlstate = code;
	return 0;
}
int pgshim_errmsg(const char *fmt, ...)
{
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(pgshim_error.message, sizeof(pgshim_error.message), fmt, ap);
	va_end(ap);
	return 0;
}
int pgshim_errdetail(const char *fmt, ...)
{
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(pgshim_error.detail, sizeof(pgshim_error.detail), fmt, ap);
	va_end(ap);
	return 0;
}
void pgshim_throw(void)
{
	if (!pgshim_handler)
	{
		fprintf(stderr, "pgshim: ERROR outside a handler: %s\n", pgshim_error.message);
		abort();
	}
	longjmp(*pgshim_handler, 1);
}

/* hash_any: Bob Jenkins' lookup3 (the published algorithm PostgreSQL's hash_any derives from).
 * Only its cost and its use as a bucket index matter here; its value is never a result. */
#define ROT(x, k) (((x) << (k)) | ((x) >> (32 - (k))))
Datum hash_any(const unsigned char *k, int keylen)
{
	uint32_t a, b, c, len = (uint32_t) keylen;
	a = b = c = 0x9e3779b9u + len + 3923095u;
	while (len >= 12)
	{
		a += k[0] | ((uint32_t) k[1] << 8) | ((uint32_t) k[2] << 16) | ((uint32_t) k[3] << 24);
		b += k[4] | ((uint32_t) k[5] << 8) | ((uint32_t) k[6] << 16) | ((uint32_t) k[7] << 24);
		c += k[8] | ((uint32_t) k[9] << 8) | ((uint32_t) k[10] << 16) | ((uint32_t) k[11] << 24);
		a -= c; a ^= ROT(c, 4); c += b;
		b -= a; b ^= ROT(a, 6); a += c;
		c -= b; c ^= ROT(b, 8); b += a;
		a -= c; a ^= ROT(c, 16); c += b;
		b -= a; b ^= ROT(a, 19); a += c;
		c -= b; c ^= ROT(b, 4); b += a;
		k += 12;
		len -= 12;
	}
	switch (len)
	{
	case 11: c += (uint32_t) k[10] << 24; /* fallthrough */
	case 10: c += (uint32_t) k[9] << 16; /* fallthrough */
	case 9: c += (uint32_t) k[8] << 8; /* fallthrough */
	case 8: b += (uint32_t) k[7] << 24; /* fallthrough */
	case 7: b += (uint32_t) k[6] << 16; /* fallthrough */
	case 6: b += (uint32_t) k[5] << 8; /* fallthrough */
	case 5: b += k[4]; /* fallthrough */
	case 4: a += (uint32_t) k[3] << 24; /* fallthrough */
	case 3: a += (uint32_t) k[2] << 16; /* fallthrough */
	case 2: a += (uint32_t) k[1] << 8; /* fallthrough */
	case 1: a += k[0];
	}
	c ^= b; c -= ROT(b, 14);
	a ^= c; a -= ROT(c, 11);
	b ^= a; b -= ROT(a, 25);
	c ^= b; c -= ROT(b, 16);
	a ^= c; a -= ROT(c, 4);
	b ^= a; b -= ROT(a, 14);
	c ^= b; c -= ROT(b, 24);
	return (Datum) c;
}

/* Compiled with -DPGSHIM_NO_REFERENCE this file is the pgshim's runtime alone (palloc, ereport, SRF helpers): what a driver
 * of the GPU glue needs when it makes no call into the reference, e.g. the planner hook's rewrite checks. */
#ifndef PGSHIM_NO_REFERENCE

/* ------------------------------------------------------------------ reference entry points */

extern Datum dna_in(PG_FUNCTION_ARGS);
extern Datum dna_out(PG_FUNCTION_ARGS);
extern Datum kmer_in(PG_FUNCTION_ARGS);
extern Datum kmer_out(PG_FUNCTION_ARGS);
extern Datum qkmer_in(PG_FUNCTION_ARGS);
extern Datum qkmer_out(PG_FUNCTION_ARGS);
extern Datum dna_length(PG_FUNCTION_ARGS);
extern Datum kmer_length(PG_FUNCTION_ARGS);
extern Datum qkmer_length(PG_FUNCTION_ARGS);
extern Datum kmer_equals(PG_FUNCTION_ARGS);
extern Datum kmer_starts_with(PG_FUNCTION_ARGS);
extern Datum kmer_starts_with_op(PG_FUNCTION_ARGS);
extern Datum kmer_containing(PG_FUNCTION_ARGS);
extern Datum kmer_contains(PG_FUNCTION_ARGS);
extern Datum generate_kmers(PG_FUNCTION_ARGS);
extern Datum kmer_hash(PG_FUNCTION_ARGS);

typedef Datum (*PGFunc)(FunctionCallInfo);

static Datum call1(PGFunc f, Datum a)
{
	FunctionCallInfoBaseData fc;
	memset(&fc, 0, sizeof(fc));
	fc.nargs = 1;
	fc.args[0].value = a;
	return f(&fc);
}
static Datum call2(PGFunc f, Datum a, Datum b)
{
	FunctionCallInfoBaseData fc;
	memset(&fc, 0, sizeof(fc));
	fc.nargs = 2;
	fc.args[0].value = a;
	fc.args[1].value = b;
	return f(&fc);
}

/* error record handed back across the plain-C boundary */
typedef struct RefError
{
	int sqlstate;	   /* 0x22503 (22P02) / 0x22001 / 0x22023 */
	int64_t row;	   /* offending row for batch calls, else -1 */
	char message[128]; /* errmsg text, verbatim from the reference */
	char detail[128];
} RefError;

static void capture(RefError *e, int64_t row)
{
	if (!e)
		return;
	e->sqlstate = pgshim_error.sqlstate;
	e->row = row;
	memcpy(e->message, pgshim_error.message, sizeof(e->message));
	memcpy(e->detail, pgshim_error.detail, sizeof(e->detail));
}

#define TRY(jb) (pgshim_handler = &(jb), setjmp(jb) == 0)

/* text -> type input function -> type output function -> text.  which: 0 dna, 1 kmer, 2 qkmer.
 * Returns 0 and writes the NUL-terminated canonical text (what psql would print) into out. */
int ref_type_roundtrip(int which, const char *text, char *out, size_t out_cap, RefError *err)
{
	jmp_buf jb;
	int rc = 1;
	size_t n = strlen(text);
	char *scratch = (char *) malloc(n + 1);
	memcpy(scratch, text, n + 1); /* the *_in functions lower-case their argument in place */
	if (TRY(jb))
	{
		PGFunc in = which == 0 ? dna_in : which == 1 ? kmer_in : qkmer_in;
		PGFunc outf = which == 0 ? dna_out : which == 1 ? kmer_out : qkmer_out;
		PGFunc lenf = which == 0 ? dna_length : which == 1 ? kmer_length : qkmer_length;
		Datum v = call1(in, PointerGetDatum(scratch));
		const char *s = (const char *) DatumGetPointer(call1(outf, v));
		int32 len = (int32) call1(lenf, v);
		if ((size_t) len != strlen(s) || strlen(s) + 1 > out_cap)
			abort();
		strcpy(out, s);
		rc = 0;
	}
	else
		capture(err, -1);
	pgshim_handler = NULL;
	arena_reset(&tl_arena);
	free(scratch);
	return rc;
}

/* SELECT * FROM generate_kmers(text::dna, k): writes the k-mers back to back (k bytes each, no
 * separators, position order) into out; *n_out = number of rows returned. */
int ref_generate_kmers(const char *text, int k, char *out, uint64_t out_cap_kmers, uint64_t *n_out,
					   RefError *err)
{
	jmp_buf jb;
	int rc = 1;
	size_t n = strlen(text);
	char *scratch = (char *) malloc(n + 1);
	memcpy(scratch, text, n + 1);
	*n_out = 0;
	if (TRY(jb))
	{
		Datum dna = call1(dna_in, PointerGetDatum(scratch));
		FunctionCallInfoBaseData fc;
		memset(&fc, 0, sizeof(fc));
		fc.nargs = 2;
		fc.args[0].value = dna;
		fc.args[1].value = (Datum) (uint32) k;
		uint64_t cnt = 0;
		for (;;)
		{
			Datum r = generate_kmers(&fc);
			if (fc.srf_done)
				break;
			struct varlena *v = (struct varlena *) DatumGetPointer(r);
			if (VARSIZE_ANY_EXHDR(v) != k)
				abort();
			if (cnt < out_cap_kmers)
				memcpy(out + cnt * (uint64_t) k, VARDATA_ANY(v), (size_t) k);
			cnt++;
		}
		*n_out = cnt;
		rc = 0;
	}
	else
		capture(err, -1);
	pgshim_handler = NULL;
	arena_reset(&tl_arena);
	free(scratch);
	return rc;
}

/* One predicate call on two text literals, exactly as SQL would evaluate it.
 *   op 0: equals(kmer a, kmer b)              a = b
 *   op 1: starts_with(kmer prefix a, kmer b)
 *   op 2: starts_with_op(kmer a, kmer prefix b)   a ^@ b
 *   op 3: contains(qkmer a, kmer b)           a @> b
 *   op 4: containing(kmer a, qkmer b)         a <@ b  */
int ref_predicate(int op, const char *a_text, const char *b_text, int *result, RefError *err)
{
	jmp_buf jb;
	int rc = 1;
	char *a = strdup(a_text), *b = strdup(b_text);
	if (TRY(jb))
	{
		PGFunc ain = (op == 3) ? qkmer_in : kmer_in;
		PGFunc bin = (op == 4) ? qkmer_in : kmer_in;
		Datum da = call1(ain, PointerGetDatum(a));
		Datum db = call1(bin, PointerGetDatum(b));
		PGFunc f = op == 0 ? kmer_equals : op == 1 ? kmer_starts_with : op == 2 ? kmer_starts_with_op
				 : op == 3 ? kmer_contains : kmer_containing;
		*result = (int) call2(f, da, db);
		rc = 0;
	}
	else
		capture(err, -1);
	pgshim_handler = NULL;
	arena_reset(&tl_arena);
	free(a);
	free(b);
	return rc;
}

/* Batched predicate over a column of fixed-length k-mers (ASCII, k bytes each, any case) against
 * one constant; out[i] in {0,1}.  op as in ref_predicate, the column is always the `kmer` side:
 *   op 0: col = const   op 1: starts_with(const, col)   op 2: col ^@ const
 *   op 3: contains(const::qkmer, col)   op 4: col <@ const::qkmer */
int ref_predicate_column(int op, const char *col, uint64_t m, int k, const char *const_text,
						 uint8_t *out, RefError *err)
{
	jmp_buf jb;
	int rc = 1;
	char *c = strdup(const_text);
	char buf[64];
	volatile uint64_t i = 0;
	if (k < 0 || k > 32)
	{
		free(c);
		return 2;
	}
	if (TRY(jb))
	{
		PGFunc cin = (op == 3 || op == 4) ? qkmer_in : kmer_in;
		Datum dc = call1(cin, PointerGetDatum(c));
		/* keep the constant alive across per-row arena resets */
		size_t csz = VARSIZE_SHORT(DatumGetPointer(dc));
		char cst[40];
		memcpy(cst, DatumGetPointer(dc), csz);
		PGFunc f = op == 0 ? kmer_equals : op == 1 ? kmer_starts_with : op == 2 ? kmer_starts_with_op
				 : op == 3 ? kmer_contains : kmer_containing;
		for (i = 0; i < m; i++)
		{
			memcpy(buf, col + i * (uint64_t) k, (size_t) k);
			buf[k] = 0;
			Datum dk = call1(kmer_in, PointerGetDatum(buf));
			Datum r;
			if (op == 0 || op == 2 || op == 4)
				r = call2(f, dk, PointerGetDatum(cst));
			else
				r = call2(f, PointerGetDatum(cst), dk);
			out[i] = (uint8_t) (r != 0);
			arena_reset(&tl_arena);
		}
		rc = 0;
	}
	else
		capture(err, (int64_t) i);
	pgshim_handler = NULL;
	arena_reset(&tl_arena);
	free(c);
	return rc;
}

/* ------------------------------------------------------------------ HashAggregate + count(*) */

typedef struct AggEntry
{
	struct varlena *key; /* datumCopy of the group key (short-header kmer varlena) */
	uint64_t count;		 /* int8inc transition state */
	uint32_t hash;
} AggEntry;

typedef struct AggTable
{
	AggEntry *slots;
	uint64_t cap, used;
	uint32_t hash_iv; /* per-worker perturbation, as PostgreSQL's TupleHashTable does for parallel
					   * aggregation (execGrouping.c, use_variable_hash_iv): without it the leader
					   * re-inserts groups in the workers' bucket order and linear probing goes quadratic */
	PgShimArena keys; /* group keys live in the aggregate's own context */
} AggTable;

static inline uint32_t agg_bucket(const AggTable *t, uint32_t h)
{
	uint32_t x = h ^ t->hash_iv; /* murmurhash32 finaliser, like execGrouping.c */
	x ^= x >> 16;
	x *= 0x85ebca6bu;
	x ^= x >> 13;
	x *= 0xc2b2ae35u;
	x ^= x >> 16;
	return x;
}

static void agg_init(AggTable *t, uint64_t cap, uint32_t iv)
{
	t->hash_iv = iv;
	uint64_t c = 1024;
	while (c < cap)
		c <<= 1;
	t->cap = c;
	t->used = 0;
	t->slots = (AggEntry *) calloc(c, sizeof(AggEntry));
	t->keys.head = NULL;
	if (!t->slots)
		abort();
}

static void agg_grow(AggTable *t);

/* lookup-or-insert through the extension's hash opclass: hash(kmer) then equals(kmer,kmer) */
static AggEntry *agg_lookup(AggTable *t, struct varlena *key, uint32_t h)
{
	if (t->used * 4 >= t->cap * 3)
		agg_grow(t);
	uint64_t mask = t->cap - 1, i = agg_bucket(t, h) & mask;
	for (;;)
	{
		AggEntry *e = &t->slots[i];
		if (!e->key)
		{
			size_t sz = VARATT_IS_SHORT(key) ? VARSIZE_SHORT(key) : VARSIZE_4B(key);
			e->key = (struct varlena *) arena_alloc(&t->keys, sz);
			memcpy(e->key, key, sz);
			e->hash = h;
			e->count = 0;
			t->used++;
			return e;
		}
		if (e->hash == h && call2(kmer_equals, PointerGetDatum(e->key), PointerGetDatum(key)))
			return e;
		i = (i + 1) & mask;
	}
}

static void agg_grow(AggTable *t)
{
	AggEntry *old = t->slots;
	uint64_t oc = t->cap;
	t->cap <<= 1;
	t->slots = (AggEntry *) calloc(t->cap, sizeof(AggEntry));
	if (!t->slots)
		abort();
	uint64_t mask = t->cap - 1;
	for (uint64_t j = 0; j < oc; j++)
		if (old[j].key)
		{
			uint64_t i = agg_bucket(t, old[j].hash) & mask;
			while (t->slots[i].key)
				i = (i + 1) & mask;
			t->slots[i] = old[j];
		}
	free(old);
}

static void agg_free(AggTable *t)
{
	free(t->slots);
	arena_free(&t->keys);
	t->slots = NULL;
}

typedef struct Worker
{
	const char *flat;
	const uint64_t *off;
	uint64_t row_lo, row_hi;
	int k;
	AggTable table;
	int failed;
	RefError err;
	uint64_t n_kmers;
} Worker;

/* Partial HashAggregate over ProjectSet(generate_kmers) over a slice of the rows */
static void *worker_main(void *arg)
{
	Worker *w = (Worker *) arg;
	jmp_buf jb;
	volatile uint64_t r = w->row_lo;
	volatile size_t cap = 1 << 16;
	char *volatile scratch = (char *) malloc(cap);
	if (TRY(jb))
	{
		for (r = w->row_lo; r < w->row_hi; r++)
		{
			uint64_t len = w->off[r + 1] - w->off[r];
			if (len + 1 > cap)
			{
				cap = len + 1;
				scratch = (char *) realloc(scratch, cap);
			}
			memcpy(scratch, w->flat + w->off[r], len);
			scratch[len] = 0;
			Datum dna = call1(dna_in, PointerGetDatum(scratch)); /* text -> dna (validates) */
			FunctionCallInfoBaseData fc;
			memset(&fc, 0, sizeof(fc));
			fc.nargs = 2;
			fc.args[0].value = dna;
			fc.args[1].value = (Datum) (uint32) w->k;
			for (;;)
			{
				Datum d = generate_kmers(&fc);
				if (fc.srf_done)
					break;
				uint32_t h = (uint32_t) call1(kmer_hash, d);
				AggEntry *e = agg_lookup(&w->table, (struct varlena *) DatumGetPointer(d), h);
				e->count++;
				w->n_kmers++;
			}
			arena_reset(&tl_arena);
		}
	}
	else
	{
		w->failed = 1;
		capture(&w->err, (int64_t) r);
	}
	pgshim_handler = NULL;
	arena_free(&tl_arena);
	free(scratch);
	return NULL;
}

typedef struct RefCounts
{
	uint64_t n_distinct;
	uint64_t n_kmers;
	int k;
	char *keys;		  /* n_distinct * k bytes, lower-case ASCII, hash-table order */
	uint64_t *counts; /* n_distinct */
} RefCounts;

/* SELECT kmer, count(*) FROM (SELECT generate_kmers(dna, k) FROM rows) GROUP BY kmer
 * rows are given as flat text + offsets (row r = flat[off[r] .. off[r+1])).  threads >= 1. */
int ref_count(const char *flat, const uint64_t *off, uint64_t n_rows, int k, int threads,
			  RefCounts *out, RefError *err)
{
	if (threads < 1)
		threads = 1;
	if ((uint64_t) threads > n_rows)
		threads = n_rows ? (int) n_rows : 1;
	Worker *ws = (Worker *) calloc((size_t) threads, sizeof(Worker));
	pthread_t *th = (pthread_t *) calloc((size_t) threads, sizeof(pthread_t));
	for (int t = 0; t < threads; t++)
	{
		ws[t].flat = flat;
		ws[t].off = off;
		ws[t].row_lo = n_rows * (uint64_t) t / (uint64_t) threads;
		ws[t].row_hi = n_rows * (uint64_t) (t + 1) / (uint64_t) threads;
		ws[t].k = k;
		agg_init(&ws[t].table, 1 << 12, (uint32_t) t * 0x9e3779b9u);
	}
	if (threads == 1)
		worker_main(&ws[0]);
	else
	{
		for (int t = 0; t < threads; t++)
			pthread_create(&th[t], NULL, worker_main, &ws[t]);
		for (int t = 0; t < threads; t++)
			pthread_join(th[t], NULL);
	}
	int rc = 0;
	int64_t first_bad = -1;
	for (int t = 0; t < threads; t++)
		if (ws[t].failed && (rc == 0 || ws[t].err.row < first_bad))
		{
			rc = 1;
			first_bad = ws[t].err.row;
			if (err)
				*err = ws[t].err;
		}
	memset(out, 0, sizeof(*out));
	out->k = k;
	if (rc == 0)
	{
		/* Finalize HashAggregate in the leader: combine partial states group by group */
		AggTable *fin = &ws[0].table;
		for (int t = 1; t < threads; t++)
		{
			AggTable *p = &ws[t].table;
			for (uint64_t j = 0; j < p->cap; j++)
				if (p->slots[j].key)
				{
					AggEntry *e = agg_lookup(fin, p->slots[j].key, p->slots[j].hash);
					e->count += p->slots[j].count;
				}
		}
		out->n_distinct = fin->used;
		out->keys = (char *) malloc(fin->used * (uint64_t) (k > 0 ? k : 1) + 1);
		out->counts = (uint64_t *) malloc((fin->used + 1) * sizeof(uint64_t));
		uint64_t n = 0;
		for (uint64_t j = 0; j < fin->cap; j++)
			if (fin->slots[j].key)
			{
				memcpy(out->keys + n * (uint64_t) k, VARDATA_ANY(fin->slots[j].key), (size_t) k);
				out->counts[n] = fin->slots[j].count;
				n++;
			}
		for (int t = 0; t < threads; t++)
			out->n_kmers += ws[t].n_kmers;
	}
	for (int t = 0; t < threads; t++)
		agg_free(&ws[t].table);
	free(ws);
	free(th);
	return rc;
}

void ref_counts_free(RefCounts *c)
{
	free(c->keys);
	free(c->counts);
	c->keys = NULL;
	c->counts = NULL;
}

/* generate_kmers over every row, no aggregation: returns the number of k-mers produced and an
 * order-independent checksum (sum of hash_any) so the work cannot be optimised away. */
int ref_generate_rows(const char *flat, const uint64_t *off, uint64_t n_rows, int k,
					  uint64_t *n_kmers, uint64_t *checksum, RefError *err)
{
	jmp_buf jb;
	int rc = 1;
	volatile uint64_t r = 0;
	uint64_t n = 0, cs = 0;
	volatile size_t cap = 1 << 16;
	char *volatile scratch = (char *) malloc(cap);
	if (TRY(jb))
	{
		for (r = 0; r < n_rows; r++)
		{
			uint64_t len = off[r + 1] - off[r];
			if (len + 1 > cap)
			{
				cap = len + 1;
				scratch = (char *) realloc(scratch, cap);
			}
			memcpy(scratch, flat + off[r], len);
			scratch[len] = 0;
			Datum dna = call1(dna_in, PointerGetDatum(scratch));
			FunctionCallInfoBaseData fc;
			memset(&fc, 0, sizeof(fc));
			fc.nargs = 2;
			fc.args[0].value = dna;
			fc.args[1].value = (Datum) (uint32) k;
			for (;;)
			{
				Datum d = generate_kmers(&fc);
				if (fc.srf_done)
					break;
				cs += (uint32_t) call1(kmer_hash, d);
				n++;
			}
			arena_reset(&tl_arena);
		}
		rc = 0;
	}
	else
		capture(err, (int64_t) r);
	pgshim_handler = NULL;
	arena_reset(&tl_arena);
	free(scratch);
	*n_kmers = n;
	*checksum = cs;
	return rc;
}

#endif /* PGSHIM_NO_REFERENCE */
