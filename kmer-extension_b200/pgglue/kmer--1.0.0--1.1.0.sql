-- kmer--1.0.0--1.1.0.sql -- additive update of the kmer extension: the GPU batch functions of kmer_gpu.c.
-- Nothing of kmer--1.0.0.sql changes (types, functions, operators and opclasses stay byte-identical); the control file can keep
-- default_version = '1.0.0':   CREATE EXTENSION kmer;  ALTER EXTENSION kmer UPDATE TO '1.1.0';
\echo Use "ALTER EXTENSION kmer UPDATE TO '1.1.0'" to load this file. \quit

-- GROUP BY kmer / count(*) over generate_kmers(dna, k) for a whole column at once (kmer.c:289-351 + kmer_hash_ops):
--   SELECT * FROM kmer_gpu_counts(ARRAY(SELECT dna FROM reads), 21)
--     ==  SELECT k.kmer, count(*) FROM reads r, generate_kmers(r.dna, 21) AS k(kmer) GROUP BY k.kmer
-- With kmer_gpu_hook.o in the module and the library preloaded (below), the stock query text is planned as this scan by itself.
CREATE FUNCTION kmer_gpu_counts(dna[], integer)
    RETURNS TABLE (kmer kmer, count bigint)
    AS 'MODULE_PATHNAME', 'kmer_gpu_counts'
    LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;

-- The k-mer abundance spectrum (count of counts) of that GROUP BY, binned on the GPU (no per-k-mer rows are materialised):
--   SELECT * FROM kmer_gpu_count_spectrum(ARRAY(SELECT dna FROM reads), 21)
--     ==  SELECT cnt AS count, count(*) AS kmers
--         FROM (SELECT count(*) AS cnt FROM reads r, generate_kmers(r.dna, 21) AS g(kmer) GROUP BY g.kmer) s
--         GROUP BY cnt ORDER BY cnt
CREATE FUNCTION kmer_gpu_count_spectrum(dna[], integer)
    RETURNS TABLE (count bigint, kmers bigint)
    AS 'MODULE_PATHNAME', 'kmer_gpu_count_spectrum'
    LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;

-- Canonical k-mers: a k-mer and its reverse complement (a<->t, c<->g, order reversed) are one group, keyed by the smaller of
-- the two texts -- the counting mode of `jellyfish count -C` and what GenomeScope expects of reads from both strands:
--   SELECT * FROM kmer_gpu_canonical_counts(ARRAY(SELECT dna FROM reads), 21)
--     ==  SELECT least(g.kmer::text COLLATE "C", reverse(translate(g.kmer::text, 'acgt', 'tgca')))::kmer AS kmer, count(*)
--         FROM reads r, generate_kmers(r.dna, 21) AS g(kmer) GROUP BY 1
CREATE FUNCTION kmer_gpu_canonical_counts(dna[], integer)
    RETURNS TABLE (kmer kmer, count bigint)
    AS 'MODULE_PATHNAME', 'kmer_gpu_canonical_counts'
    LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;

-- The abundance spectrum of that canonical GROUP BY:
--   SELECT * FROM kmer_gpu_canonical_count_spectrum(ARRAY(SELECT dna FROM reads), 21)
--     ==  SELECT cnt AS count, count(*) AS kmers
--         FROM (SELECT count(*) AS cnt FROM reads r, generate_kmers(r.dna, 21) AS g(kmer)
--               GROUP BY least(g.kmer::text COLLATE "C", reverse(translate(g.kmer::text, 'acgt', 'tgca')))) s
--         GROUP BY cnt ORDER BY cnt
CREATE FUNCTION kmer_gpu_canonical_count_spectrum(dna[], integer)
    RETURNS TABLE (count bigint, kmers bigint)
    AS 'MODULE_PATHNAME', 'kmer_gpu_canonical_count_spectrum'
    LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;

-- equals / starts_with / contains over a column of k-mers against one constant (kmer.c:226-285):
--   element i of the result:  op 0  kmer[i] = $2      op 1  kmer[i] ^@ $2      op 2  $2::qkmer @> kmer[i]
CREATE FUNCTION kmer_gpu_match(kmer[], text, integer)
    RETURNS SETOF boolean
    AS 'MODULE_PATHNAME', 'kmer_gpu_match'
    LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;

-- The planner hook (kmer_gpu_hook.c) is installed by the module's _PG_init, i.e. when the shared library is loaded into the
-- backend.  PostgreSQL loads an extension's library lazily, at the first call of one of its C functions -- which for a plain
-- `SELECT ... generate_kmers(dna, 21) ... GROUP BY` happens at execution, AFTER that statement was planned.  To have the first
-- statement of a session offloaded too, preload the library:
--   ALTER SYSTEM SET session_preload_libraries = 'kmer';     -- or shared_preload_libraries; or per role / database
-- SET kmer.gpu_offload = off  plans the stock query the stock way again.
