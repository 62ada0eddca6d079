/* tests/c/hook_driver.c -- runs the planner hook of the GPU glue (kmer-extension_b200/pgglue/kmer_gpu_hook.c, SURVEY 8 f4) on
 * analyzed Query trees built by hand the way PostgreSQL's parser builds them for the reference's stock counting queries
 * (kmer-tests.sql:1162-1181 TEST 13.1 and the configs' `SELECT kmer, count(*) FROM (SELECT generate_kmers(dna, k) ...) GROUP BY kmer`):
 *
 *   structure (no GPU)  : the three stock shapes are rewritten into a function scan on kmer_gpu_counts(...), the ORDER BY / LIMIT
 *                         variants keep their clauses, and every query that is NOT exactly such a count (HAVING, another
 *                         aggregate, count(kmer), FILTER, WHERE on the outer level, non-constant k, another SRF, a second output
 *                         column, two grouping columns, WITH ORDINALITY, LIMIT in the subquery, the GUC off, the glue's SQL function
 *                         missing) is handed to the next planner untouched;
 *   --exec (GPU)        : the REWRITTEN tree is executed by a tiny stand-in executor over a fake `reads` table -- the ARRAY
 *                         sublink scanned, kmer_gpu_counts (kmer_gpu.c) driven through the fmgr shim -- and its rows must equal,
 *                         datum for datum and count for count, what the ORIGINAL query computes with the reference's own
 *                         generate_kmers (oracle/_ref) under a sort + group -- built with -DPGSHIM_NO_REFERENCE, with the
 *                         C oracle's generate_kmers instead (tests/c/expected_kmers.h).
 * Built and run by tests/test_hook.py.  Exit code 0 = all as expected. */
#include "postgres.h"
#include "fmgr.h"
#include "funcapi.h"
#include "catalog/pg_type.h"
#include "nodes/parsenodes.h"
#include "nodes/makefuncs.h"
#include "optimizer/planner.h"
#include "utils/array.h"

extern void _PG_init(void);
extern Datum kmer_gpu_counts(PG_FUNCTION_ARGS);
extern void pgshim_catalog_reset(void);
extern void pgshim_catalog_add_type(const char *name, Oid oid, Oid array_oid);
extern void pgshim_catalog_add_func(const char *name, int nargs, const Oid *args, Oid oid);
extern bool pgshim_set_bool_guc(const char *name, bool value);

enum { DNA_OID = 70001, DNA_ARRAY_OID = 70002, KMER_OID = 70003, KMER_ARRAY_OID = 70004, GENERATE_KMERS_OID = 70010, GPU_COUNTS_OID = 70011,
	   OTHER_SRF_OID = 70012, READS_RELID = 16384, COUNT_STAR_OID = 2803, COUNT_ANY_OID = 2147, MIN_OID = 2145, OP_ID_IS_EVEN = 99001 };

static void fill_catalog(int with_gpu_function)
{
	Oid a[2];
	pgshim_catalog_reset();
	pgshim_catalog_add_type("dna", DNA_OID, DNA_ARRAY_OID);
	pgshim_catalog_add_type("kmer", KMER_OID, KMER_ARRAY_OID);
	a[0] = DNA_OID; a[1] = INT4OID;
	pgshim_catalog_add_func("generate_kmers", 2, a, GENERATE_KMERS_OID);
	if (with_gpu_function)
	{
		a[0] = DNA_ARRAY_OID;
		pgshim_catalog_add_func("kmer_gpu_counts", 2, a, GPU_COUNTS_OID);
	}
}

/* ------------------------------------------------------------------ building analyzed trees */
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

static Const *int4_const(int v)
{
	Const *c = makeNode(Const);
	c->consttype = INT4OID; c->consttypmod = -1; c->constlen = 4; c->constvalue = (Datum) v; c->constbyval = true; c->location = -1;
	return c;
}

static Const *dna_const(const char *text)
{
	Const *c = makeNode(Const);
	c->consttype = DNA_OID; c->consttypmod = -1; c->constlen = -1; c->location = -1;
	c->constvalue = PointerGetDatum(make_varlena(text, (int) strlen(text), 0)); /* what dna_in returns, kmer.c:92-93 */
	return c;
}

static FuncExpr *srf_call(Oid funcid, Node *dna, Node *k)
{
	FuncExpr *f = makeFuncExpr(funcid, KMER_OID, list_make2(dna, k), InvalidOid, InvalidOid, COERCE_EXPLICIT_CALL);
	f->funcretset = true;
	return f;
}

static Aggref *count_agg(Oid fn, int star, Node *arg)
{
	Aggref *a = makeNode(Aggref);
	a->aggfnoid = fn; a->aggtype = INT8OID; a->aggstar = star != 0; a->aggkind = 'n'; a->location = -1;
	if (arg) a->args = list_make1(makeTargetEntry((Expr *) arg, 1, NULL, false));
	return a;
}

static RangeTblEntry *reads_rte(const char *alias)
{
	RangeTblEntry *r = makeNode(RangeTblEntry);
	r->rtekind = RTE_RELATION; r->relid = READS_RELID; r->relkind = 'r'; r->perminfoindex = 1; r->inh = true; r->inFromCl = true;
	r->eref = makeAlias(alias, list_make2(makeString("id"), makeString("dna")));
	if (strcmp(alias, "reads")) r->alias = makeAlias(alias, NIL);
	return r;
}

static SortGroupClause *sgc(Index ref)
{
	SortGroupClause *s = makeNode(SortGroupClause);
	s->tleSortGroupRef = ref; s->eqop = 98001; s->sortop = 98002; s->hashable = true;
	return s;
}

static Query *select_query(void)
{
	Query *q = makeNode(Query);
	q->commandType = CMD_SELECT; q->querySource = QSRC_ORIGINAL; q->canSetTag = true;
	return q;
}

static FromExpr *from_refs(int n, Node *quals)
{
	List *l = NIL;
	for (int i = 1; i <= n; i++)
	{
		RangeTblRef *r = makeNode(RangeTblRef);
		r->rtindex = i;
		l = lappend(l, r);
	}
	return makeFromExpr(l, quals);
}

static Node *where_id_is_even(void)   /* WHERE id % 2 = 0, as one opaque operator node the stand-in executor understands */
{
	OpExpr *o = makeNode(OpExpr);
	o->opno = OP_ID_IS_EVEN;
	o->args = list_make1(makeVar(1, 1, INT4OID, -1, InvalidOid, 0));
	return (Node *) o;
}

/* the outer level shared by all shapes: SELECT <kmer col>, count(*) ... GROUP BY <kmer col> */
static void outer_level(Query *q, int kmer_varno)
{
	TargetEntry *t1 = makeTargetEntry((Expr *) makeVar(kmer_varno, 1, KMER_OID, -1, InvalidOid, 0), 1, "kmer", false);
	TargetEntry *t2 = makeTargetEntry((Expr *) count_agg(COUNT_STAR_OID, 1, NULL), 2, "count", false);
	t1->ressortgroupref = 1;
	q->targetList = list_make2(t1, t2);
	q->groupClause = list_make1(sgc(1));
	q->hasAggs = true;
}

/* S2: SELECT kmer, count(*) FROM (SELECT generate_kmers(dna, k) AS kmer FROM reads [WHERE id % 2 = 0]) s GROUP BY kmer */
static Query *stock_s2(int k, int with_where)
{
	Query *sq = select_query(), *q = select_query();
	RangeTblEntry *s = makeNode(RangeTblEntry);
	sq->rtable = list_make1(reads_rte("reads"));
	sq->rteperminfos = list_make1(makeString("perminfo(reads)"));
	sq->jointree = from_refs(1, with_where ? where_id_is_even() : NULL);
	sq->targetList = list_make1(makeTargetEntry((Expr *) srf_call(GENERATE_KMERS_OID, (Node *) makeVar(1, 2, DNA_OID, -1, InvalidOid, 0), (Node *) int4_const(k)), 1, "kmer", false));
	sq->hasTargetSRFs = true;
	s->rtekind = RTE_SUBQUERY; s->subquery = sq; s->inFromCl = true;
	s->alias = makeAlias("s", NIL);
	s->eref = makeAlias("s", list_make1(makeString("kmer")));
	q->rtable = list_make1(s);
	q->jointree = from_refs(1, NULL);
	outer_level(q, 1);
	return q;
}

/* S3: SELECT k.kmer, count(*) FROM reads r, generate_kmers(r.dna, k) AS k(kmer) GROUP BY k.kmer */
static Query *stock_s3(int k)
{
	Query *q = select_query();
	RangeTblEntry *f = makeNode(RangeTblEntry);
	RangeTblFunction *rtf = makeNode(RangeTblFunction);
	rtf->funcexpr = (Node *) srf_call(GENERATE_KMERS_OID, (Node *) makeVar(1, 2, DNA_OID, -1, InvalidOid, 0), (Node *) int4_const(k));
	rtf->funccolcount = 1;
	f->rtekind = RTE_FUNCTION; f->functions = list_make1(rtf); f->lateral = true; f->inFromCl = true;
	f->alias = makeAlias("k", list_make1(makeString("kmer")));
	f->eref = makeAlias("k", list_make1(makeString("kmer")));
	q->rtable = list_make2(reads_rte("r"), f);
	q->rteperminfos = list_make1(makeString("perminfo(reads)"));
	q->jointree = from_refs(2, NULL);
	outer_level(q, 2);
	return q;
}

/* S1: SELECT k.kmer, count(*) FROM generate_kmers('ACGTACGT'::dna, 4) AS k(kmer) GROUP BY k.kmer   (TEST 13.1) */
static Query *stock_s1(const char *dna, int k)
{
	Query *q = select_query();
	RangeTblEntry *f = makeNode(RangeTblEntry);
	RangeTblFunction *rtf = makeNode(RangeTblFunction);
	rtf->funcexpr = (Node *) srf_call(GENERATE_KMERS_OID, (Node *) dna_const(dna), (Node *) int4_const(k));
	rtf->funccolcount = 1;
	f->rtekind = RTE_FUNCTION; f->functions = list_make1(rtf); f->inFromCl = true;
	f->alias = makeAlias("k", list_make1(makeString("kmer")));
	f->eref = makeAlias("k", list_make1(makeString("kmer")));
	q->rtable = list_make1(f);
	q->jointree = from_refs(1, NULL);
	outer_level(q, 1);
	return q;
}

/* SELECT t.kmer, t.count FROM (<counting query>) t ORDER BY 2 DESC */
static Query *wrap_in_select(Query *inner)
{
	Query *q = select_query();
	RangeTblEntry *t = makeNode(RangeTblEntry);
	TargetEntry *t1 = makeTargetEntry((Expr *) makeVar(1, 1, KMER_OID, -1, InvalidOid, 0), 1, "kmer", false);
	TargetEntry *t2 = makeTargetEntry((Expr *) makeVar(1, 2, INT8OID, -1, InvalidOid, 0), 2, "count", false);
	t->rtekind = RTE_SUBQUERY; t->subquery = inner; t->inFromCl = true;
	t->alias = makeAlias("t", NIL);
	t->eref = makeAlias("t", list_make2(makeString("kmer"), makeString("count")));
	t2->ressortgroupref = 1;
	q->rtable = list_make1(t);
	q->jointree = from_refs(1, NULL);
	q->targetList = list_make2(t1, t2);
	q->sortClause = list_make1(sgc(1));
	return q;
}

/* ------------------------------------------------------------------ structure checks */
static int prev_hook_calls;
static PlannedStmt *previous_hook(Query *parse, const char *qs, int co, ParamListInfo bp)
{
	prev_hook_calls++;
	return standard_planner(parse, qs, co, bp);
}

static Query *plan(Query *q)
{
	PlannedStmt *p = planner_hook(q, "<stock query>", 0, NULL);
	return p->pgshim_query;
}

static int is_rewritten(const Query *q, Node **array_arg, Const **k_arg)
{
	if (q->hasAggs || q->groupClause != NIL || list_length(q->rtable) != 1) return 0;
	RangeTblEntry *r = (RangeTblEntry *) linitial(q->rtable);
	if (r->rtekind != RTE_FUNCTION || list_length(r->functions) != 1 || r->lateral || r->funcordinality) return 0;
	RangeTblFunction *rtf = (RangeTblFunction *) linitial(r->functions);
	if (!IsA(rtf->funcexpr, FuncExpr) || rtf->funccolcount != 2) return 0;
	FuncExpr *f = (FuncExpr *) rtf->funcexpr;
	if (f->funcid != GPU_COUNTS_OID || !f->funcretset || f->funcresulttype != RECORDOID || list_length(f->args) != 2) return 0;
	if (list_length(r->eref->colnames) != 2 || strcmp(strVal(linitial(r->eref->colnames)), "kmer") || strcmp(strVal(lsecond(r->eref->colnames)), "count")) return 0;
	if (list_length(q->jointree->fromlist) != 1 || ((RangeTblRef *) linitial(q->jointree->fromlist))->rtindex != 1 || q->jointree->quals) return 0;
	/* output columns: plain Vars of the function scan, same order, names and resnos as before */
	TargetEntry *t1 = (TargetEntry *) linitial(q->targetList), *t2 = (TargetEntry *) lsecond(q->targetList);
	Var *v1 = (Var *) t1->expr, *v2 = (Var *) t2->expr;
	if (!IsA(v1, Var) || v1->varno != 1 || v1->varattno != 1 || v1->vartype != KMER_OID || strcmp(t1->resname, "kmer") || t1->resno != 1) return 0;
	if (!IsA(v2, Var) || v2->varno != 1 || v2->varattno != 2 || v2->vartype != INT8OID || strcmp(t2->resname, "count") || t2->resno != 2) return 0;
	*array_arg = (Node *) linitial(f->args);
	*k_arg = (Const *) lsecond(f->args);
	return 1;
}

static int failures;
#define CHECK(cond, what) do { int ok__ = (cond); printf("[hook] %-100s %s\n", what, ok__ ? "ok" : "MISMATCH"); if (!ok__) failures++; } while (0)

static void structure_tests(void)
{
	Node *arr;
	Const *kc;

	fill_catalog(1);
	/* S2, with and without a WHERE in the subquery */
	for (int w = 0; w < 2; w++)
	{
		Query *q = stock_s2(21, w);
		Query *sq = ((RangeTblEntry *) linitial(q->rtable))->subquery;
		Node *quals = sq->jointree->quals;
		Const *k_before = (Const *) lsecond(((FuncExpr *) ((TargetEntry *) linitial(sq->targetList))->expr)->args);
		Query *p = plan(q);
		int ok = p == q && is_rewritten(p, &arr, &kc) && kc == k_before && IsA(arr, SubLink) && ((SubLink *) arr)->subLinkType == ARRAY_SUBLINK &&
				 ((SubLink *) arr)->subselect == (Node *) sq && p->hasSubLinks && !sq->hasTargetSRFs && sq->jointree->quals == quals &&
				 list_length(sq->targetList) == 1 && list_length(sq->rteperminfos) == 1;
		if (ok)
		{
			Var *d = (Var *) ((TargetEntry *) linitial(sq->targetList))->expr;
			ok = IsA(d, Var) && d->varno == 1 && d->varattno == 2 && d->vartype == DNA_OID && ((RangeTblEntry *) linitial(sq->rtable))->relid == READS_RELID;
		}
		ok = ok && ((TargetEntry *) linitial(p->targetList))->ressortgroupref == 0;
		CHECK(ok, w ? "S2 (subquery with WHERE): function scan on kmer_gpu_counts(ARRAY(SELECT dna FROM reads WHERE ...), 21)"
					: "S2: SELECT kmer, count(*) FROM (SELECT generate_kmers(dna, 21) ...) GROUP BY kmer -> function scan");
	}
	/* S2 ... ORDER BY count(*) DESC LIMIT 5 and ORDER BY kmer: the clauses stay and still point at their target entries */
	{
		Query *q = stock_s2(21, 0);
		((TargetEntry *) lsecond(q->targetList))->ressortgroupref = 2;
		q->sortClause = list_make1(sgc(2));
		q->limitCount = (Node *) int4_const(5);
		Query *p = plan(q);
		CHECK(is_rewritten(p, &arr, &kc) && list_length(p->sortClause) == 1 && ((SortGroupClause *) linitial(p->sortClause))->tleSortGroupRef == 2 &&
				  ((TargetEntry *) lsecond(p->targetList))->ressortgroupref == 2 && p->limitCount != NULL,
			  "S2 ... ORDER BY count(*) DESC LIMIT 5: rewritten, sort and limit kept");
		q = stock_s2(21, 0);
		q->sortClause = list_make1(sgc(1));
		p = plan(q);
		CHECK(is_rewritten(p, &arr, &kc) && ((TargetEntry *) linitial(p->targetList))->ressortgroupref == 1 && list_length(p->sortClause) == 1,
			  "S2 ... ORDER BY kmer: rewritten, the k-mer column keeps its sort reference");
	}
	/* S3 */
	{
		Query *q = stock_s3(31);
		RangeTblEntry *rel = (RangeTblEntry *) linitial(q->rtable);
		Query *p = plan(q);
		int ok = is_rewritten(p, &arr, &kc) && IsA(arr, SubLink) && (int) kc->constvalue == 31 && p->rteperminfos == NIL;
		if (ok)
		{
			Query *in = (Query *) ((SubLink *) arr)->subselect;
			Var *d = (Var *) ((TargetEntry *) linitial(in->targetList))->expr;
			ok = IsA(in, Query) && in->commandType == CMD_SELECT && list_length(in->rtable) == 1 && linitial(in->rtable) == (void *) rel &&
				 list_length(in->rteperminfos) == 1 && IsA(d, Var) && d->varno == 1 && d->varattno == 2 && !in->hasAggs && !in->hasTargetSRFs &&
				 list_length(in->jointree->fromlist) == 1;
		}
		CHECK(ok, "S3: FROM reads r, generate_kmers(r.dna, 31) AS k(kmer) GROUP BY k.kmer -> ARRAY(SELECT r.dna FROM reads r)");
	}
	/* S1 (TEST 13.1) */
	{
		Query *q = stock_s1("ACGTACGT", 4);
		Query *p = plan(q);
		int ok = is_rewritten(p, &arr, &kc) && IsA(arr, ArrayExpr) && ((ArrayExpr *) arr)->array_typeid == DNA_ARRAY_OID &&
				 ((ArrayExpr *) arr)->element_typeid == DNA_OID && list_length(((ArrayExpr *) arr)->elements) == 1 && !p->hasSubLinks;
		CHECK(ok, "S1 (TEST 13.1): FROM generate_kmers('ACGTACGT'::dna, 4) AS k(kmer) -> kmer_gpu_counts(ARRAY['ACGTACGT'::dna], 4)");
	}
	/* the counting query as a sub-select of a larger statement: SELECT kmer, count FROM (<S2>) t ORDER BY 2 DESC */
	{
		Query *in = stock_s2(21, 1), *top = wrap_in_select(in);
		Query *p = plan(top);
		RangeTblEntry *t = (RangeTblEntry *) linitial(p->rtable);
		CHECK(p == top && t->rtekind == RTE_SUBQUERY && t->subquery == in && is_rewritten(in, &arr, &kc) && !top->hasAggs &&
				  list_length(top->sortClause) == 1,
			  "S2 as a sub-select in FROM of a larger statement: the inner level is rewritten, the outer one untouched");
	}
	CHECK(prev_hook_calls >= 7, "the planner hook that was installed before _PG_init is still called (hook chain)");

	/* ---- queries that must reach the planner untouched ---- */
#define UNTOUCHED(q, what) do { Query *q__ = (q); int n__ = list_length(q__->rtable); RTEKind k__ = ((RangeTblEntry *) linitial(q__->rtable))->rtekind; \
		Query *p__ = plan(q__); CHECK(p__ == q__ && p__->hasAggs && p__->groupClause != NIL && list_length(p__->rtable) == n__ && \
		((RangeTblEntry *) linitial(p__->rtable))->rtekind == k__ && !is_rewritten(p__, &arr, &kc), what); } while (0)
	Query *q;
	q = stock_s2(21, 0); q->havingQual = (Node *) count_agg(COUNT_STAR_OID, 1, NULL);
	UNTOUCHED(q, "not rewritten: HAVING count(*) > 1");
	q = stock_s2(21, 0); q->targetList = lappend(q->targetList, makeTargetEntry((Expr *) count_agg(MIN_OID, 0, (Node *) makeVar(1, 1, KMER_OID, -1, InvalidOid, 0)), 3, "min", false));
	UNTOUCHED(q, "not rewritten: a third output column with another aggregate");
	q = stock_s2(21, 0); ((TargetEntry *) lsecond(q->targetList))->expr = (Expr *) count_agg(COUNT_ANY_OID, 0, (Node *) makeVar(1, 1, KMER_OID, -1, InvalidOid, 0));
	UNTOUCHED(q, "not rewritten: count(kmer) instead of count(*)");
	q = stock_s2(21, 0); ((Aggref *) ((TargetEntry *) lsecond(q->targetList))->expr)->aggfilter = (Expr *) where_id_is_even();
	UNTOUCHED(q, "not rewritten: count(*) FILTER (WHERE ...)");
	q = stock_s2(21, 0); ((Aggref *) ((TargetEntry *) lsecond(q->targetList))->expr)->aggdistinct = list_make1(sgc(1));
	UNTOUCHED(q, "not rewritten: count(DISTINCT ...)");
	q = stock_s2(21, 0); q->jointree->quals = where_id_is_even();
	UNTOUCHED(q, "not rewritten: WHERE on the outer level");
	q = stock_s2(21, 0);
	lsecond(((FuncExpr *) ((TargetEntry *) linitial(((RangeTblEntry *) linitial(q->rtable))->subquery->targetList))->expr)->args) = makeVar(1, 1, INT4OID, -1, InvalidOid, 0);
	UNTOUCHED(q, "not rewritten: k is a column, not a constant");
	q = stock_s2(21, 0); ((FuncExpr *) ((TargetEntry *) linitial(((RangeTblEntry *) linitial(q->rtable))->subquery->targetList))->expr)->funcid = OTHER_SRF_OID;
	UNTOUCHED(q, "not rewritten: another set-returning function");
	q = stock_s2(21, 0);
	{
		Query *sq = ((RangeTblEntry *) linitial(q->rtable))->subquery;
		sq->targetList = lappend(sq->targetList, makeTargetEntry((Expr *) makeVar(1, 1, INT4OID, -1, InvalidOid, 0), 2, "id", false));
	}
	UNTOUCHED(q, "not rewritten: the subquery has a second output column");
	q = stock_s2(21, 0); ((RangeTblEntry *) linitial(q->rtable))->subquery->limitCount = (Node *) int4_const(10);
	UNTOUCHED(q, "not rewritten: LIMIT inside the subquery");
	q = stock_s2(21, 0);
	{
		TargetEntry *t3 = makeTargetEntry((Expr *) makeVar(1, 1, KMER_OID, -1, InvalidOid, 0), 3, "kmer2", false);
		t3->ressortgroupref = 3;
		q->targetList = lappend(q->targetList, t3);
		q->groupClause = lappend(q->groupClause, sgc(3));
	}
	UNTOUCHED(q, "not rewritten: two grouping columns");
	q = stock_s2(21, 0); q->distinctClause = list_make1(sgc(1));
	UNTOUCHED(q, "not rewritten: SELECT DISTINCT");
	q = stock_s3(21); ((RangeTblEntry *) lsecond(q->rtable))->funcordinality = true;
	UNTOUCHED(q, "not rewritten: generate_kmers(...) WITH ORDINALITY");
	q = stock_s3(21); q->jointree->quals = where_id_is_even();
	UNTOUCHED(q, "not rewritten: S3 with a WHERE clause");
	q = stock_s1("ACGTACGT", 4); ((Const *) linitial(((FuncExpr *) ((RangeTblFunction *) linitial(((RangeTblEntry *) linitial(q->rtable))->functions))->funcexpr)->args))->constisnull = true;
	UNTOUCHED(q, "not rewritten: generate_kmers(NULL, 4)");
	pgshim_set_bool_guc("kmer.gpu_offload", false);
	UNTOUCHED(stock_s2(21, 0), "not rewritten: SET kmer.gpu_offload = off");
	pgshim_set_bool_guc("kmer.gpu_offload", true);
	fill_catalog(0);
	UNTOUCHED(stock_s2(21, 0), "not rewritten: kmer_gpu_counts(dna[], integer) is not installed");
	fill_catalog(1);
	{
		Query *ins = stock_s2(21, 0);
		ins->commandType = CMD_INSERT;
		Query *p = plan(ins);
		CHECK(p == ins && p->hasAggs, "not rewritten: not a SELECT");
	}
}

/* ------------------------------------------------------------------ the rewritten tree executed (GPU) */
static uint64_t rng_state = 0x2545F4914F6CDD1DULL;
static uint32_t rnd(void)
{
	rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17;
	return (uint32_t) (rng_state >> 32);
}

typedef struct FakeTable { int n; struct varlena **dna; } FakeTable; /* reads(id = row number, dna) */

static int row_qualifies(Node *quals, int id)
{
	if (!quals) return 1;
	return ((OpExpr *) quals)->opno == OP_ID_IS_EVEN ? id % 2 == 0 : 0;
}

/* what the ORIGINAL query computes: generate_kmers over every qualifying row (the reference, or the C oracle), sort, group */
static size_t reference_groups(const FakeTable *t, Node *quals, struct varlena *const_dna, int k, Item **out)
{
	Item *want = NULL;
	size_t n = 0, cap = 0, g = 0;
	int rows = const_dna ? 1 : t->n;
	for (int r = 0; r < rows; r++)
	{
		if (!const_dna && !row_qualifies(quals, r)) continue;
		struct varlena *src = const_dna ? const_dna : t->dna[r];
		int len = VARSIZE_ANY_EXHDR(src);
		char *low = (char *) palloc((Size) len + 1);
		for (int i = 0; i < len; i++) low[i] = (char) (VARDATA_ANY(src)[i] | 0x20); /* dna_in lower-cases, kmer.c:28-29 */
		want = expected_kmers(want, &n, &cap, low, len, k);
	}
	qsort(want, n, sizeof(Item), cmp_item);
	for (size_t i = 0; i < n; i++)
	{
		if (g && !memcmp(want[g - 1].bytes, want[i].bytes, 40)) want[g - 1].count++;
		else want[g++] = want[i];
	}
	*out = want;
	return g;
}

/* the stand-in executor for the REWRITTEN tree: Function Scan on kmer_gpu_counts(<array expression>, k), projected through the target list */
static size_t execute_rewritten(const Query *q, const FakeTable *t, Item **out)
{
	RangeTblFunction *rtf = (RangeTblFunction *) linitial(((RangeTblEntry *) linitial(q->rtable))->functions);
	FuncExpr *f = (FuncExpr *) rtf->funcexpr;
	Node *a0 = (Node *) linitial(f->args);
	int k = (int) ((Const *) lsecond(f->args))->constvalue;
	ArrayType *arr;
	if (IsA(a0, SubLink))
	{
		/* ARRAY(SELECT <dna column> FROM reads [WHERE ...]): a sequential scan of the fake table */
		Query *in = (Query *) ((SubLink *) a0)->subselect;
		Var *col = (Var *) ((TargetEntry *) linitial(in->targetList))->expr;
		if (col->varattno != 2 || ((RangeTblEntry *) linitial(in->rtable))->relid != READS_RELID) { printf("executor: unexpected inner query\n"); exit(2); }
		arr = (ArrayType *) palloc(sizeof(ArrayType) + (size_t) t->n * sizeof(Datum));
		arr->nelems = 0;
		arr->elemtype = DNA_OID;
		for (int r = 0; r < t->n; r++)
			if (row_qualifies(in->jointree->quals, r)) arr->elems[arr->nelems++] = PointerGetDatum(t->dna[r]);
	}
	else
	{
		ArrayExpr *ae = (ArrayExpr *) a0;
		arr = (ArrayType *) palloc(sizeof(ArrayType) + sizeof(Datum));
		arr->nelems = 1;
		arr->elemtype = ae->element_typeid;
		arr->elems[0] = ((Const *) linitial(ae->elements))->constvalue;
	}
	FunctionCallInfoBaseData fc;
	memset(&fc, 0, sizeof(fc));
	fc.nargs = 2;
	fc.args[0].value = PointerGetDatum(arr);
	fc.args[1].value = (Datum) k;
	Item *got = NULL;
	size_t n = 0, cap = 0;
	int kmer_att = ((Var *) ((TargetEntry *) linitial(q->targetList))->expr)->varattno, count_att = ((Var *) ((TargetEntry *) lsecond(q->targetList))->expr)->varattno;
	for (;;)
	{
		Datum d = kmer_gpu_counts(&fc);
		if (fc.srf_done) break;
		HeapTuple tup = (HeapTuple) DatumGetPointer(d);
		if (n == cap) { cap = cap ? cap * 2 : 4096; got = (Item *) realloc(got, cap * sizeof(Item)); }
		struct varlena *v = (struct varlena *) DatumGetPointer(tup->values[kmer_att - 1]);
		memset(&got[n], 0, sizeof(Item));
		memcpy(got[n].bytes, v, (size_t) VARSIZE_SHORT(v));
		got[n].count = DatumGetInt64(tup->values[count_att - 1]);
		n++;
	}
	qsort(got, n, sizeof(Item), cmp_item);
	*out = got;
	return n;
}

static void exec_case(const char *what, Query *q, const FakeTable *t, Node *orig_quals, struct varlena *const_dna, int k)
{
	Item *want, *got;
	size_t g = reference_groups(t, orig_quals, const_dna, k, &want);
	Query *p = plan(q);
	Node *arr;
	Const *kc;
	if (!p->hasAggs && p->groupClause == NIL && ((RangeTblEntry *) linitial(p->rtable))->rtekind == RTE_SUBQUERY)
		p = ((RangeTblEntry *) linitial(p->rtable))->subquery;   /* a pass-through outer level: execute the level below it */
	if (!is_rewritten(p, &arr, &kc)) { CHECK(0, what); return; }
	size_t n = execute_rewritten(p, t, &got);
	int ok = n == g;
	for (size_t i = 0; ok && i < g; i++) ok = !memcmp(got[i].bytes, want[i].bytes, 40) && got[i].count == want[i].count;
	char line[200];
	snprintf(line, sizeof(line), "%s: rewritten plan on the GPU == original query via " EXPECTED_SOURCE " (%zu/%zu groups)", what, n, g);
	CHECK(ok, line);
	free(want); free(got);
}

static void exec_tests(void)
{
	FakeTable t;
	t.n = 3000;
	t.dna = (struct varlena **) palloc(sizeof(struct varlena *) * (size_t) t.n);
	char buf[400];
	for (int r = 0; r < t.n; r++)
	{
		int len = 40 + (int) (rnd() % 300);
		if (r % 9 == 0) rng_state = 77 + (uint64_t) (r % 63); /* some reads repeat: counts above 1 */
		for (int i = 0; i < len; i++) buf[i] = "ACGTacgt"[rnd() & 7];
		t.dna[r] = make_varlena(buf, len, r & 1);            /* both header forms, as on disk / in memory */
	}
	fill_catalog(1);
	exec_case("S2 k=21", stock_s2(21, 0), &t, NULL, NULL, 21);
	exec_case("S2 k=31 WHERE id % 2 = 0", stock_s2(31, 1), &t, where_id_is_even(), NULL, 31);
	exec_case("S2 k=22 inside a larger statement", wrap_in_select(stock_s2(22, 1)), &t, where_id_is_even(), NULL, 22);
	exec_case("S3 k=5", stock_s3(5), &t, NULL, NULL, 5);
	exec_case("S3 k=32", stock_s3(32), &t, NULL, NULL, 32);
	{
		Const *c = dna_const("ACGTACGT");
		Query *q = stock_s1("ACGTACGT", 4);
		exec_case("S1 TEST 13.1 generate_kmers('ACGTACGT', 4)", q, &t, NULL, (struct varlena *) DatumGetPointer(c->constvalue), 4);
	}
}

int main(int argc, char **argv)
{
	planner_hook = previous_hook;      /* some other extension's hook, installed first */
	_PG_init();
	structure_tests();
	if (argc > 1 && !strcmp(argv[1], "--exec"))
		exec_tests();
	printf("[hook] %s\n", failures ? "FAILED" : "all ok");
	return failures ? 1 : 0;
}
