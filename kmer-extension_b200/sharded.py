"""Sharded k-mer counting and matching: one process per GPU; counting splits the rows across ranks (one all-to-all or none), matching splits the k-mer column (no data-path collective: class ShardedMatcher at the end).

The reference has no distributed path (its only parallelism is PostgreSQL's parallel query); this is
the multi-GPU form of `SELECT kmer, count(*) ... GROUP BY kmer` over generate_kmers (kmer.c:289-351):

  1. every rank partitions ITS rows' k-mers into the same global minimizer buckets
     (kmer_cuda_dev_shard_partition),
  2. bucket b is owned by rank b // buckets_per_rank.  On GPUs (exchange="pull", the default) there is NO separate
     exchange step: the ranks' send blocks are opened in every process once (CUDA IPC), a tiny all-reduce on the
     stream tells every rank that all partitions are done, and the owner's split kernel reads its (bucket, source)
     segments straight out of the sources' memory over NVLink (kmer_cuda_dev_shard_count_peers).
     exchange="nccl" (and the CPU plumbing tests): ONE all-to-all (equal splits) moves every segment to its owner,
     a second small one the fill counts (optionally, chunks=2, the rows are partitioned in two pieces and the
     exchange of the first piece runs on a side stream while the second piece is being partitioned),
  3. every owner counts its buckets on chip (kmer_cuda_dev_shard_count*).

Identical k-mers share a minimizer, hence a bucket, hence an owner, so the per-rank results are
disjoint and the GROUP BY result is their concatenation.  k <= 13 uses the dense 4^k table instead:
all-reduce(sum) of the per-rank tables, every rank emits the bins it owns.

`torch.distributed` is the transport (NCCL on GPUs; gloo in the CPU plumbing tests, where the engine is
a stand-in).  The library itself never communicates.
"""
from __future__ import annotations

import contextlib

import torch
import torch.distributed as dist

KMER_ERR_CAPACITY = 20   # include/kmer_cuda.h


class ShardedCounter:
    def __init__(self, engine, group=None, device=None, chunks=None, exchange=None):
        self.eng = engine
        self.chunks = chunks       # pieces a rank's rows are partitioned in (None: 1)
        self.exchange = exchange   # "pull" | "nccl" | None: pull on GPUs when the engine can (KMER_SHARD_EXCHANGE overrides)
        self._pull = None          # {"block": tensor, "addr": [device address of every rank's block], "opened": [bases]}
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.device = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        self._bufs = {}
        self.last_plan = None
        self._xbytes = 0
        self.last_phases = []      # (name, ms) of the last count when the engine's profiling is on

    @property
    def last_exchange_bytes(self) -> int:
        """Bytes this rank's records and fill counts put on the links in the last count."""
        if callable(self._xbytes):
            self._xbytes = self._xbytes()
        return self._xbytes

    @last_exchange_bytes.setter
    def last_exchange_bytes(self, v):
        self._xbytes = v

    # ------------------------------------------------------------------ helpers
    def _buf(self, name, nbytes, dtype=torch.uint8):
        item = torch.empty((), dtype=dtype).element_size()
        n = (nbytes + item - 1) // item
        t = self._bufs.get(name)
        if t is None or t.numel() < n or t.dtype != dtype:
            t = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self._bufs[name] = t
        return t[:n]

    def _use_pull(self, chunks) -> bool:
        import os
        mode = self.exchange or os.environ.get("KMER_SHARD_EXCHANGE") or "pull"
        return (mode == "pull" and chunks == 1 and self.world > 1 and self.device.type == "cuda"
                and hasattr(self.eng, "ipc_export"))

    def _pull_block(self, nbytes: int):
        """This rank's send block (records, then fills) and every rank's view of it.  (Re)allocated when the plan outgrows it:
        the size follows from the plan alone, so every rank takes this branch in the same call -- it is collective."""
        st = self._pull
        if st is not None and st["block"].numel() >= nbytes:
            return st
        torch.cuda.synchronize(self.device)
        self.close()
        block = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        try:
            mine = self.eng.ipc_export(block)
        except Exception:                       # e.g. an allocator that does not hand out cudaMalloc memory
            mine = None
        everyone = [None] * self.world
        dist.all_gather_object(everyone, mine, group=self.group)
        addr, opened, ok = [], [], all(e is not None for e in everyone)
        if ok:
            try:
                for r, (h, o) in enumerate(everyone):
                    if r == self.rank:
                        addr.append(block.data_ptr())
                    else:
                        base = self.eng.ipc_open(h)
                        opened.append(base)
                        addr.append(base + o)
            except Exception:                   # no peer access between two of the GPUs
                ok = False
        self._pull = {"block": block, "addr": addr, "opened": opened,
                      "token": torch.zeros(1, dtype=torch.int32, device=self.device)}
        # every rank has opened every block (nobody proceeds, and could free its block, before that) -- or all fall back together
        if not self._allreduce_int(1 if ok else 0, dist.ReduceOp.MIN):
            self.close()
            self.exchange = "nccl"
            return None
        return self._pull

    def close(self):
        """Unmaps the peers' send blocks (collective in spirit: call it on every rank before the process group goes away)."""
        st, self._pull = self._pull, None
        if st is not None:
            for base in st["opened"]:
                try:
                    self.eng.ipc_close(base)
                except Exception:
                    pass

    def _allreduce_int(self, value: int, op=dist.ReduceOp.SUM) -> int:
        if self.world == 1:
            return int(value)
        t = torch.tensor([int(value)], dtype=torch.int64, device=self.device)
        dist.all_reduce(t, op=op, group=self.group)
        return int(t.item())

    @staticmethod
    def _find_cut(d_off, n_rows: int):
        """A row index near the middle whose first base sits on a 16-byte boundary of the column (or None)."""
        if n_rows < 64:
            return None
        mid = n_rows // 2
        window = d_off[mid: min(mid + 256, n_rows)]
        hit = ((window % 16) == 0).nonzero()
        if hit.numel() == 0:
            return None
        return mid + int(hit[0].item())

    def _phases(self):
        return list(self.eng.phases()) if hasattr(self.eng, "phases") else []

    def _agree(self, exc):
        """All ranks raise if any rank failed with an INPUT error (the lowest failing rank's error text wins on that rank
        only).  Returns True if some rank only ran out of room (KMER_ERR_CAPACITY: segment / spill list / output overflow on
        skewed input) and nothing worse happened anywhere: every rank then takes the exact fallback together."""
        code = 0
        if exc is not None:
            code = 1 if getattr(exc, "status", None) == KMER_ERR_CAPACITY else 2
        worst = self._allreduce_int(code, dist.ReduceOp.MAX)
        if worst == 2:
            if exc is not None and code == 2:
                raise exc
            raise RuntimeError("sharded count aborted: another rank reported an input error")
        return worst == 1

    # ------------------------------------------------------------------ the operation
    def count(self, d_seq, n_bases: int, d_off, n_rows: int, k: int, d_pairs, total_kmers: int | None = None, d_uniq=None):
        """Counts this rank's rows together with all other ranks' rows.

        d_pairs: int64 [capacity, 2] on this rank; returns (n_distinct_here, n_kmers_counted_here, info dict).
        d_uniq (int64 [capacity], k >= 14): split result format -- groups with count 1 come back as bare codes in d_uniq
        (info["n_unique"] of them), n_distinct_here then counts the pairs only.
        Collective: every rank of the group must call it with the same k."""
        eng = self.eng
        local_kmers = eng.max_kmers(n_bases, n_rows, k)
        if total_kmers is None:
            total_kmers = self._allreduce_int(local_kmers)
        if k <= 13:
            return self._count_dense(d_seq, n_bases, d_off, n_rows, k, d_pairs, total_kmers)

        def owner_count(plan, pst, recv_recs, recv_fill, recs_bytes):
            if pst is not None:
                rb, bpr = plan.recs_bytes_per_peer, plan.buckets_per_rank
                eng.dev_shard_count_peers(plan, [a + self.rank * rb for a in pst["addr"]],
                                          [a + recs_bytes + self.rank * bpr * 8 for a in pst["addr"]], d_uniq, d_pairs)
            elif d_uniq is not None:
                eng.dev_shard_count_split(plan, recv_recs, recv_fill, d_uniq, d_pairs)
            else:
                eng.dev_shard_count(plan, recv_recs, recv_fill, d_pairs)
        r = self._exchange_and_count(d_seq, n_bases, d_off, n_rows, k, total_kmers, owner_count)
        if r is None:                     # skewed input: some segment or spill list ran out of room -- exact fallback, all ranks together
            return self._count_fallback(d_seq, n_bases, d_off, n_rows, k, d_pairs, total_kmers)
        return int(r.n_distinct), int(r.n_kmers), {"tier2_kmers": int(r.n_tier2), "plan": self.last_plan,
                                                  "n_unique": int(getattr(r, "n_unique", 0)), "fallback": False}

    def _exchange_and_count(self, d_seq, n_bases, d_off, n_rows, k, total_kmers, owner_count):
        """The minimizer exchange (k >= 14) and this rank's owner count, owner_count(plan, pull state or None, recv_recs,
        recv_fill, recs_bytes) -- one of the library's dev_shard_count* calls.  Returns the count's dev_finish result, or None
        when some rank ran out of room (KMER_ERR_CAPACITY): every rank then takes the exact fallback together."""
        eng = self.eng
        # chunks=2 partitions the rows in two pieces and exchanges the first on a side stream while the second is being
        # partitioned.  Measured on 2xB200 it LOSES (18.8 vs 17.9 ms/step: two launches and host round trips per step, and
        # the exchange slows the partition kernel it runs beside), so it is opt-in.
        chunks = self.chunks if self.chunks is not None else 1
        # every rank must cut its rows in the same number of pieces: a piece starts on a 16-byte boundary of the column
        cut = None
        if chunks == 2:
            cut = self._find_cut(d_off, n_rows)
            ok = self._allreduce_int(0 if cut is None else 1, dist.ReduceOp.MIN)
            if not ok:
                chunks, cut = 1, None
        if chunks == 1:
            plan = eng.shard_plan(max(total_kmers, 1), k, self.world)
        else:
            plan = eng.shard_plan(max(total_kmers, 1), k, self.world, chunks)
        self.last_plan = plan
        recs_bytes = plan.recs_bytes_per_peer * self.world       # one piece
        fill_words = plan.buckets_per_rank * self.world
        pull = self._use_pull(chunks)
        pst = self._pull_block(recs_bytes + fill_words * 8) if pull else None
        pull = pst is not None
        if pull:
            send_recs = pst["block"][:recs_bytes]
            send_fill = pst["block"][recs_bytes:recs_bytes + fill_words * 8].view(torch.int64)
            recv_recs = recv_fill = None
        else:
            send_recs = self._buf("send_recs", recs_bytes * chunks)
            send_fill = self._buf("send_fill", fill_words * 8 * chunks, torch.int64)
            recv_recs = self._buf("recv_recs", recs_bytes * chunks) if self.world > 1 else send_recs
            recv_fill = self._buf("recv_fill", fill_words * 8 * chunks, torch.int64) if self.world > 1 else send_fill
        pieces = [(0, n_rows)] if chunks == 1 else [(0, cut), (cut, n_rows)]
        exc = None
        phases = []
        timed = self.device.type == "cuda" and getattr(eng, "profiling", False)
        comm = None
        if self.world > 1 and self.device.type == "cuda":
            if getattr(self, "_comm_stream", None) is None:
                self._comm_stream = torch.cuda.Stream(device=self.device)
            comm = self._comm_stream
        a2a_events = []
        chained = chunks == 1          # partition -> exchange -> count on the device without a host round trip in between
        for ci, (r0, r1) in enumerate(pieces):
            sr = send_recs[ci * recs_bytes:(ci + 1) * recs_bytes]
            sf = send_fill[ci * fill_words:(ci + 1) * fill_words]
            try:
                if chunks == 1:
                    eng.dev_shard_partition(d_seq, n_bases, d_off, n_rows, plan, sr, sf)
                else:
                    b0 = int(d_off[r0].item())
                    b1 = int(d_off[r1].item())
                    eng.dev_shard_partition(d_seq[b0:], b1 - b0, d_off[r0:r1 + 1] - b0, r1 - r0, plan, sr, sf)
                    eng.dev_finish()      # the piece is partitioned (host waits): its exchange may start
                    phases += self._phases()
            except Exception as e:  # input error or segment overflow on this rank
                exc = exc or e
            if pull:
                # every rank's partition is done when this tiny all-reduce has run on the stream (no host wait): the owners then
                # read the segments where they are.  The sources do not touch their blocks again before the all-reduce that ends
                # this call, which every rank joins only after its own count has finished.
                dist.all_reduce(pst["token"], group=self.group)
            elif self.world > 1:
                rr = recv_recs[ci * recs_bytes:(ci + 1) * recs_bytes]
                rf = recv_fill[ci * fill_words:(ci + 1) * fill_words]
                if comm is not None:
                    comm.wait_stream(torch.cuda.current_stream())      # the exchange follows the partition kernel on the device
                    with torch.cuda.stream(comm):
                        if timed and not chained:
                            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                            e0.record()
                        dist.all_to_all_single(rf, sf, group=self.group)
                        dist.all_to_all_single(rr, sr, group=self.group)
                        if timed and not chained:
                            e1.record()
                            a2a_events.append((e0, e1))
                else:
                    dist.all_to_all_single(rf, sf, group=self.group)
                    dist.all_to_all_single(rr, sr, group=self.group)
        if comm is not None:
            torch.cuda.current_stream().wait_stream(comm)
            if timed and not chained:
                torch.cuda.synchronize()
                phases.append(("all_to_all", sum(a.elapsed_time(b) for a, b in a2a_events)))
        if pull:       # what the other GPUs' split kernels read from here: the filled part of their segments (evaluated on demand)
            own = slice(self.rank * plan.buckets_per_rank, (self.rank + 1) * plan.buckets_per_rank)
            rec_bytes = plan.rec_bytes

            def sent(fill=send_fill, own=own, rec_bytes=rec_bytes):
                low = fill & 0xffffffff
                return int((low.sum() - low[own].sum()).item()) * rec_bytes + (fill.numel() - (own.stop - own.start)) * 8
            self.last_exchange_bytes = sent
        elif self.world > 1:
            self.last_exchange_bytes = int(recs_bytes + fill_words * 8) * chunks * (self.world - 1) // self.world
        else:
            self.last_exchange_bytes = 0
        # The count is queued right behind the exchange; ONE finish reports the partition's findings (input errors, a
        # segment overflow) together with the count's, and ONE all-reduce makes every rank act on the same outcome.
        r = None
        if exc is None:
            try:
                owner_count(plan, pst if pull else None, recv_recs, recv_fill, recs_bytes)
                r = eng.dev_finish()
            except Exception as e:        # no rank may be left waiting in a collective
                exc = e
        code = 0 if exc is None else (1 if getattr(exc, "status", None) == KMER_ERR_CAPACITY else 2)
        if self.world > 1:
            t = torch.tensor([1 if code == 2 else 0, 1 if code == 1 else 0, int(r.n_kmers) if r is not None else 0], dtype=torch.int64,
                             device=self.device)
            dist.all_reduce(t, group=self.group)
            n_input_err, n_capacity, counted = (int(x) for x in t.tolist())
        else:
            n_input_err, n_capacity, counted = int(code == 2), int(code == 1), int(r.n_kmers) if r is not None else 0
        if n_input_err:
            if code == 2:
                raise exc
            raise RuntimeError("sharded count aborted: another rank reported an input error")
        if n_capacity:
            return None
        phases += self._phases()
        self.last_phases = phases
        if counted != total_kmers:
            raise RuntimeError(f"sharded count lost k-mers: counted {counted}, expected {total_kmers}")
        return r

    def spectrum(self, d_seq, n_bases: int, d_off, n_rows: int, k: int, hist_len: int = 65536, total_kmers: int | None = None):
        """The abundance spectrum (count of counts) of this rank's rows together with all other ranks' rows; collective.

        Returns (hist, tail, info), the SAME on every rank: hist int64 [hist_len] -- hist[c] = k-mers counted exactly c times --
        and tail int64 [n, 2], the (code, count) groups with count >= hist_len, ranks' tails in rank order.  Every owner bins its
        own groups (disjoint across ranks), then one all-reduce sums the histograms and an all-gather joins the tails."""
        eng = self.eng
        if total_kmers is None:
            total_kmers = self._allreduce_int(eng.max_kmers(n_bases, n_rows, k))
        hist = self._buf("spec_hist", hist_len * 8, torch.int64)
        tail = self._buf("spec_tail", max(total_kmers // hist_len, 1) * 16, torch.int64).view(-1, 2)
        info = {"plan": None, "fallback": False, "tier2_kmers": 0}
        if k <= 13:
            owned = self._buf("spec_pairs", ((1 << (2 * k)) + self.world - 1) // self.world * 16, torch.int64).view(-1, 2)
            nd, _, _ = self._count_dense(d_seq, n_bases, d_off, n_rows, k, owned, total_kmers)
            n_tail = self._pairs_spectrum(owned, nd, hist, tail)
        else:
            def owner_count(plan, pst, recv_recs, recv_fill, recs_bytes):
                rb, bpr = plan.recs_bytes_per_peer, plan.buckets_per_rank
                if pst is not None:
                    src_r = [a + self.rank * rb for a in pst["addr"]]
                    src_f = [a + recs_bytes + self.rank * bpr * 8 for a in pst["addr"]]
                else:                         # the receive buffers: source s's segments at s * recs_bytes_per_peer
                    n_src = recv_fill.numel() // bpr
                    src_r = [recv_recs.data_ptr() + s * rb for s in range(n_src)]
                    src_f = [recv_fill.data_ptr() + s * bpr * 8 for s in range(n_src)]
                eng.dev_shard_count_spectrum(plan, src_r, src_f, hist, tail)
            r = self._exchange_and_count(d_seq, n_bases, d_off, n_rows, k, total_kmers, owner_count)
            if r is None:                 # the exact fallback: the owners' merged tables, then their spectrum
                owned = self._buf("spec_pairs", (int(total_kmers / self.world * 1.3) + 65536) * 16, torch.int64).view(-1, 2)
                nd, _, info = self._count_fallback(d_seq, n_bases, d_off, n_rows, k, owned, total_kmers)
                n_tail = self._pairs_spectrum(owned, nd, hist, tail)
            else:
                n_tail = int(r.n_distinct)
                info = {"plan": self.last_plan, "fallback": False, "tier2_kmers": int(r.n_tier2)}
        hist_all, tail_all = self._combine_spectrum(hist, tail[:n_tail])
        return hist_all, tail_all, info

    def _pairs_spectrum(self, pairs, n, hist, tail) -> int:
        exc, r = None, None
        try:
            self.eng.dev_pairs_spectrum(pairs, n, hist, tail)
            r = self.eng.dev_finish()
        except Exception as e:
            exc = e
        if self._agree(exc) or exc is not None:
            raise exc if exc is not None else RuntimeError("sharded spectrum aborted: another rank's tail buffer is too small")
        return int(r.n_distinct)

    def _combine_spectrum(self, hist, tail):
        """The owners' spectra -> the job's: histograms summed, tails gathered (sizes first), on every rank."""
        hist = hist.clone()
        if self.world == 1:
            return hist, tail.clone()
        dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=self.group)
        n = torch.tensor([tail.shape[0]], dtype=torch.int64, device=self.device)
        sizes = [torch.zeros_like(n) for _ in range(self.world)]
        dist.all_gather(sizes, n, group=self.group)
        sizes = [int(x.item()) for x in sizes]
        pad = torch.zeros((max(max(sizes), 1), 2), dtype=torch.int64, device=self.device)
        pad[:tail.shape[0]] = tail
        parts = [torch.empty_like(pad) for _ in range(self.world)]
        dist.all_gather(parts, pad, group=self.group)
        return hist, torch.cat([p[:m] for p, m in zip(parts, sizes)])

    def _count_fallback(self, d_seq, n_bases, d_off, n_rows, k, d_pairs, total_kmers):
        """Exact on ANY input (HashAggregate never refuses rows, kmer-tests.sql:1208-1213): every rank counts its own rows with
        the single-GPU counter (tiers 2/3 absorb any skew), then the tables are merged by owner = hash(k-mer) % world: the
        ranks' tables are broadcast in turn and every rank keeps the groups it owns.  Slower than the minimizer exchange
        (whole tables travel), only taken when that one ran out of room."""
        eng = self.eng
        cap_local = max(eng.max_kmers(n_bases, n_rows, k), 1)
        local = self._buf("fb_local", cap_local * 16, torch.int64).view(-1, 2)
        exc, n_loc = None, 0
        try:
            eng.dev_count(d_seq, n_bases, d_off, n_rows, k, local)
            n_loc = int(eng.dev_finish().n_distinct)
        except Exception as e:
            exc = e
        if self._agree(exc):
            raise exc if exc is not None else RuntimeError("sharded count aborted: another rank ran out of memory")
        counts = [n_loc]
        if self.world > 1:
            t = torch.tensor([n_loc], dtype=torch.int64, device=self.device)
            all_n = [torch.zeros_like(t) for _ in range(self.world)]
            dist.all_gather(all_n, t, group=self.group)
            counts = [int(x.item()) for x in all_n]
        # the owner hash spreads DISTINCT k-mers evenly whatever their counts: this rank owns about sum/world groups
        eng.dev_merge_begin(int(sum(counts) / self.world * 1.3) + 65536)
        buf = self._buf("fb_bcast", max(max(counts), 1) * 16, torch.int64).view(-1, 2) if self.world > 1 else local
        for src in range(self.world):
            if counts[src] == 0:
                continue
            if self.world > 1:
                if src == self.rank:
                    buf[:counts[src]].copy_(local[:counts[src]])
                dist.broadcast(buf[:counts[src]], src, group=self.group)
            eng.dev_merge_add(buf, counts[src], self.rank, self.world)
        exc, r = None, None
        try:
            eng.dev_merge_emit(k, d_pairs)
            r = eng.dev_finish()
        except Exception as e:
            exc = e
        if self._agree(exc) or exc is not None:
            raise exc if exc is not None else RuntimeError("sharded count aborted: another rank's output buffer is too small")
        self.last_exchange_bytes = int(sum(counts) * 16)
        self.last_phases = []
        counted = self._allreduce_int(int(r.n_kmers))
        if counted != total_kmers:
            raise RuntimeError(f"sharded fallback lost k-mers: counted {counted}, expected {total_kmers}")
        return int(r.n_distinct), int(r.n_kmers), {"tier2_kmers": 0, "plan": None, "n_unique": 0, "fallback": True}

    def _count_dense(self, d_seq, n_bases, d_off, n_rows, k, d_pairs, total_kmers):
        eng = self.eng
        table = self._buf("dense", 8 << (2 * k), torch.int64)
        exc = None
        try:
            eng.dev_dense_table(d_seq, n_bases, d_off, n_rows, k, table)
            eng.dev_finish()
        except Exception as e:
            exc = e
        if self._agree(exc):
            raise exc
        if self.world > 1:
            dist.all_reduce(table, op=dist.ReduceOp.SUM, group=self.group)
            self.last_exchange_bytes = int(table.numel() * 8)
        r = None
        try:
            eng.dev_dense_emit(table, k, self.rank, self.world, d_pairs)
            r = eng.dev_finish()
        except Exception as e:            # output buffer too small on this rank: all ranks raise together
            exc = e
        if self._agree(exc) or exc is not None:
            raise exc if exc is not None else RuntimeError("sharded dense count aborted: another rank's output buffer is too small")
        counted = self._allreduce_int(int(r.n_kmers))
        if counted != total_kmers:
            raise RuntimeError(f"sharded dense count lost k-mers: counted {counted}, expected {total_kmers}")
        return int(r.n_distinct), int(r.n_kmers), {"tier2_kmers": 0, "plan": None}


class ShardedMatcher:
    """Batched equals / starts_with / contains over a k-mer column that is sharded across the ranks (SURVEY 8e: "matching is
    embarrassingly parallel over k-mers: shard M, replicate patterns, no collective").

    The reference evaluates these predicates one (constant, k-mer) pair per fmgr call (kmer_equals kmer.c:226-245,
    kmer_starts_with* kmer.c:248-265, kmer_contains / kmer_containing kmer.c:268-285); here every rank holds the slice
    [lo, hi) of the column given by `slice_of` -- slices start on a multiple of 32 k-mers, so the ranks' rows of the P x M bit
    matrix are whole 32-bit words and concatenate without shifting -- and the constants are replicated.  A rank's bits never
    leave it (the caller reads its slice of every row back, or filters its slice of the rows); the only communication is one
    all-reduce of P hit counters plus an error flag, on the stream, so that a rank that fails does not leave the others waiting.
    """

    def __init__(self, engine, group=None, device=None):
        self.eng = engine
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.device = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        self._acc = None

    @staticmethod
    def slice_of(m_total: int, rank: int, world: int):
        """k-mers [lo, hi) of the column that `rank` matches: even split, cut points on multiples of 32."""
        def cut(r):
            return m_total if r >= world else (m_total * r // world) & ~31
        return cut(rank), cut(rank + 1)

    @staticmethod
    def words_per_row(m: int) -> int:
        return (m + 31) // 32

    def match(self, op, d_codes, m_local: int, k: int, consts, d_bits, d_hits, d_lens=None, ops=None, stream=None):
        """This rank's slice against the replicated constants.  d_bits: int32[P * words_per_row(m_local)] (this rank's words
        of every row), d_hits: int64[P] -- on return the hit counts over the WHOLE column (summed over the ranks).
        Returns the local dev_finish result.  Raises on every rank if any rank failed."""
        consts = [consts] if isinstance(consts, str) else list(consts)
        P = len(consts)
        if self._acc is None or self._acc.numel() < P + 1:
            self._acc = torch.zeros(P + 1, dtype=torch.int64, device=self.device)
        acc = self._acc[:P + 1]
        # the counters are copied and reduced on the stream the kernels run on (NCCL takes torch's current stream)
        on = torch.cuda.stream(stream) if (stream is not None and self.device.type == "cuda") else contextlib.nullcontext()
        exc = None
        with on:
            try:
                self.eng.dev_match(op, d_codes, m_local, k, consts, d_bits, d_hits, d_lens=d_lens, ops=ops, stream=stream)
            except Exception as e:     # constants are replicated, so a bad constant raises everywhere; a device error may not
                exc = e
            if exc is None:
                acc[:P].copy_(d_hits[:P])
                acc[P:].zero_()
            else:
                acc.zero_()
                acc[P:].fill_(1)
            if self.world > 1:
                dist.all_reduce(acc, group=self.group)
            res = None
            try:
                res = self.eng.dev_finish(stream)
            except Exception as e:
                exc = exc or e
            failed = int(acc[P].item())
            if exc is not None:
                raise exc
            if failed:
                raise RuntimeError(f"sharded match: {failed} other rank(s) failed")
            d_hits[:P].copy_(acc[:P])
        return res

    def gather_bits(self, d_bits, m_local: int, m_total: int, P: int):
        """The whole P x words_per_row(m_total) bit matrix on every rank (tests / small results; the product path keeps a
        rank's words on the rank).  Rows are the concatenation of the ranks' words in rank order."""
        wl = self.words_per_row(m_local)
        if self.world == 1:
            return d_bits[:P * wl].view(P, wl).clone()
        cuts = [self.slice_of(m_total, r, self.world) for r in range(self.world)]
        wmax = max(self.words_per_row(hi - lo) for lo, hi in cuts)
        mine = torch.zeros((P, wmax), dtype=d_bits.dtype, device=d_bits.device)
        if wl:
            mine[:, :wl] = d_bits[:P * wl].view(P, wl)
        parts = [torch.empty_like(mine) for _ in range(self.world)]
        dist.all_gather(parts, mine, group=self.group)
        return torch.cat([parts[r][:, :self.words_per_row(hi - lo)] for r, (lo, hi) in enumerate(cuts)], dim=1)
