"""The ingest pipeline the spec's write path describes (README.md:1507-1583, resolved per
SURVEY.md §0.2 C1): CDC -> SHA-256 -> exact dedup -> DEFLATE of first occurrences, on one GPU
(`Ingest`) or on byte-range shards of one stream across GPUs (`ShardedIngest`)."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import torch

from . import sharding
from .api import Context, file_offsets
from .config import CDCConfig, SimConfig


@dataclass
class IngestResult:
    cuts: torch.Tensor        # int64 (uint64 bit patterns) exclusive end offsets, local to the shard buffer
    digests: torch.Tensor     # uint8 [n, 32]
    canon: torch.Tensor       # int64 [n]: index (global id when sharded) of the first equal chunk
    is_first: torch.Tensor    # bool [n]
    select: torch.Tensor      # int64 [m] chunks that were compressed
    blob: torch.Tensor        # uint8 packed zlib streams
    offsets: torch.Tensor     # int64 [m + 1]
    entry: int = 0            # offset of the first owned chunk (sharded)
    id_base: int = 0          # global id of local chunk 0 (sharded)
    base: Optional[torch.Tensor] = None           # L4: int64 [n] base chunk of every chunk stored as a delta, else -1
    delta_blob: Optional[torch.Tensor] = None     # L4: uint8 packed deltas (chunk order)
    delta_offsets: Optional[torch.Tensor] = None  # L4: int64 [n + 1]
    file_chunk: Optional[torch.Tensor] = None     # files: int64 [F + 1] index of each file's first chunk (run(files=...))
    known: Optional[torch.Tensor] = None          # known=: int64 [m] archive slot each stream was copied from, or -1
    stats: Optional[dict] = None                  # known=: streams / bytes copied, streams / raw bytes compressed

    @property
    def n_chunks(self) -> int:
        return int(self.cuts.numel())


class Ingest:
    def __init__(self, ctx: Context, cdc: CDCConfig = CDCConfig(), zdict=b"", level: int = 6):
        self.ctx, self.cdc, self.level = ctx, cdc, level
        self.zdict = ctx.stage(zdict) if not isinstance(zdict, torch.Tensor) else zdict

    def select_first(self, first_u8: torch.Tensor) -> torch.Tensor:
        n = first_u8.numel()
        sel = self.ctx.empty(max(n, 1), torch.int64)
        m = C.c_uint64(0)
        self.ctx.check(self.ctx.lib.hmse_dedup_select(self.ctx.h, first_u8.data_ptr(), n, sel.data_ptr(), n, C.byref(m),
                                                      self.ctx.stream))
        return sel[:m.value]

    def similarity_delta(self, d: torch.Tensor, cuts: torch.Tensor, first: torch.Tensor, sim: SimConfig, min_votes: int = 4,
                         start0: int = 0):
        """The L4 stage (README.md:1553-1570): MinHash -> band keys -> buckets -> base selection -> delta coding with
        the 20 % rule.  Returns (base int64[n], delta blob, delta offsets int64[n+1]).  `start0`: offset of chunk 0
        in `d` (a shard whose first owned chunk does not start at 0)."""
        ctx = self.ctx
        # Only first occurrences are hashed (the spec computes MinHash after the exact-dedup miss, README.md:1553-1556).
        # Duplicates never head a bucket (their first occurrence has the same keys and a smaller index), so selecting
        # bases among the first occurrences alone, in their compacted index space, gives the same bases.
        sel = self.select_first(first.view(torch.uint8))
        m = sel.numel()
        keys = ctx.lsh_keys(ctx.minhash(d, cuts, sim, start0=start0, select=sel), sim)
        band, key, ids = ctx.lsh_buckets(keys)
        ones = torch.ones(m, dtype=torch.uint8, device=ctx.tdev)
        base_u = ctx.delta_bases(band, key, ids, m, sim.bands, ones, min_votes)
        base = torch.full((cuts.numel(),), -1, dtype=torch.int64, device=ctx.tdev)
        base[sel] = torch.where(base_u >= 0, sel[base_u.clamp(min=0)], base_u)
        dblob, doffs = ctx.delta_encode(d, cuts, base, start0=start0)
        return base, dblob, doffs

    def open_known(self, known, compress: bool):
        """The archive of run(known=...), opened: a Reader is used as it is, an Archive is opened for the call; None when
        the archive stores no chunk (nothing can be known).  Raises ValueError when its dictionary differs
        from this ingest's or nothing is compressed."""
        from .archive import Reader
        if not compress:
            raise ValueError("known= needs compress=True: it decides which streams are copied instead of compressed")
        ar = known.ar if isinstance(known, Reader) else known
        if bytes(ar.zdict) != bytes(self.zdict.cpu().numpy()):
            raise ValueError("the archive's dictionary differs from the ingest's")
        if ar.n_unique == 0:
            return None
        return known if isinstance(known, Reader) else Reader(known, self.ctx)

    def compress_known(self, rd, d: torch.Tensor, cuts: torch.Tensor, digests: torch.Tensor, sel: torch.Tensor, start0: int = 0,
                       out: Optional[torch.Tensor] = None, ctx: Optional[Context] = None):
        """(blob, offsets, known, stats): the selected chunks compressed against the opened archive `rd`
        (hmse_compress_known) - blob and offsets are what Context.compress returns."""
        ctx = ctx or self.ctx
        if rd is None:
            blob, offs = ctx.compress(d, cuts, sel, self.zdict, self.level, start0=start0, out=out)
            starts = torch.cat([torch.full((1,), start0, dtype=torch.int64, device=cuts.device), cuts[:-1]])
            raw = int((cuts - starts)[sel].sum()) if sel.numel() else 0
            kn = torch.full((sel.numel(),), -1, dtype=torch.int64, device=ctx.tdev)
            return blob, offs, kn, dict(copied=0, copied_bytes=0, compressed=int(sel.numel()), compressed_raw_bytes=raw)
        blob, offs, kn, st4 = ctx.compress_known(rd.src(), d, cuts, digests, sel, self.zdict, self.level, start0=start0, out=out)
        return blob, offs, kn, dict(copied=st4[0], copied_bytes=st4[1], compressed=st4[2], compressed_raw_bytes=st4[3])

    def run(self, d: torch.Tensor, compress: bool = True, l4: Optional[SimConfig] = None, min_votes: int = 4,
            files=None, known=None) -> IngestResult:
        """l4: also run the similarity layer; first occurrences that keep a delta are not compressed (`select` lists
        the chunks of the chunk store only) and `base` / `delta_blob` / `delta_offsets` describe the deltas.
        files: the sizes of the files `d` holds back to back (a sequence or an integer tensor, zeros allowed).  Every
        file is then chunked on its own (hmse_chunk_files): no chunk spans two files, so equal files give equal chunks
        wherever they sit, and `file_chunk` records where each file's chunks begin.  Everything after chunking runs
        unchanged over the one chunk list.
        known: an archive (`Archive`, opened for the call, or an opened `Reader`) whose streams are reused: a stored chunk
        whose digest and raw length the archive holds takes the archive's stream instead of being compressed
        (hmse_compress_known).  Every field equals the run without `known` when the archive was written by this encoder at
        the same level and dictionary; `known` (int64 [m]) names the archive slot each stream came from (-1: compressed)
        and `stats` counts what was copied and compressed."""
        ctx = self.ctx
        rd = self.open_known(known, compress) if known is not None else None
        d = ctx.stage(d)     # unchanged when it is aligned and has slack behind it; re-staged otherwise
        file_chunk = None
        if files is None:
            cuts = ctx.chunk(d, self.cdc)
        else:
            cuts, file_chunk = ctx.chunk_files(d, file_offsets(files, d.numel(), ctx), self.cdc)
        digests = ctx.digest(d, cuts)
        canon, first = ctx.dedup(digests)
        base = dblob = doffs = None
        stored = first
        if l4 is not None and cuts.numel():
            base, dblob, doffs = self.similarity_delta(d, cuts, first, l4, min_votes)
            stored = first & (base < 0)
        sel = self.select_first(stored.view(torch.uint8))
        kn = stats = None
        if known is not None:
            blob, offs, kn, stats = self.compress_known(rd, d, cuts, digests, sel)
        elif compress:
            blob, offs = ctx.compress(d, cuts, sel, self.zdict, self.level)
        else:
            blob, offs = ctx.empty(0, torch.uint8), ctx.empty(1, torch.int64).zero_()
        return IngestResult(cuts, digests, canon, first, sel, blob, offs, base=base, delta_blob=dblob, delta_offsets=doffs,
                            file_chunk=file_chunk, known=kn, stats=stats)


@dataclass
class HostIngestResult:
    """What IngestStream leaves in (pinned) host memory; same meaning as IngestResult, absolute offsets."""
    cuts: torch.Tensor        # int64 [n]
    digests: torch.Tensor     # uint8 [n, 32]
    canon: torch.Tensor       # int64 [n]
    offsets: torch.Tensor     # int64 [m + 1]
    blob: torch.Tensor        # uint8
    h2d_bytes: int = 0
    d2h_bytes: int = 0
    known: Optional[torch.Tensor] = None   # run(known=...): int64 [m] archive slot each stream was copied from, or -1
    stats: Optional[dict] = None           # run(known=...): summed over the pieces

    @property
    def n_chunks(self) -> int:
        return int(self.cuts.numel())

    @property
    def is_first(self) -> torch.Tensor:
        return self.canon == torch.arange(self.canon.numel(), dtype=torch.int64)

    @property
    def select(self) -> torch.Tensor:
        return torch.nonzero(self.is_first).view(-1)


class IngestStream(Ingest):
    """Host-to-host ingest of one stream in pieces (the spec's Core 0 I/O stage feeding the
    pipeline, README.md:141-145): piece k+1 is copied host->device while piece k is chunked,
    hashed, deduplicated against everything seen so far (hmse_dedup_begin/append) and
    compressed, and the results of piece k-1 travel device->host - three CUDA streams (four with `overlap`: the
    chunking, hashing and deduplication of piece k+1 then run on their own stream, host thread and hmse_ctx beside the
    compression of piece k).
    A chunk that straddles a piece boundary is resolved with the next piece (the boundary rule of
    hmse_chunk_resolve), so cuts, digests, canon and streams equal the one-shot `Ingest.run`.
    Pieces grow from piece_bytes/16 to piece_bytes and shrink again at the end of the stream: the
    first kernels start after a short copy and little is left to copy out after the last one."""

    def __init__(self, ctx: Context, cdc: CDCConfig = CDCConfig(), zdict=b"", level: int = 6, piece_bytes: int = 1 << 30,
                 overlap: bool = False):
        super().__init__(ctx, cdc, zdict, level)
        # overlap: run the front stage (cuts, digests, dedup) of the next piece on its own thread/stream/ctx beside the
        # compression.  Measured on B200: no gain (152.0 -> 151.3 ms per 4 GB) - the persistent parse CTAs hold every
        # SM's registers, so the front kernels only run where the compression kernels would have; off by default.
        self.overlap = overlap
        self.ctx2 = None           # second hmse_ctx (own scratch and mailbox) for the compression side when overlapping
        self.s_front = None
        if piece_bytes % 16 or piece_bytes < 4 * cdc.max_size:
            raise ValueError("piece_bytes must be a multiple of 16 and >= 4 * max_size")
        self.piece = int(piece_bytes)
        self.s_h2d = torch.cuda.Stream(ctx.tdev)
        self.s_d2h = torch.cuda.Stream(ctx.tdev)
        self._dbufs = [None, None]   # device input buffers: the stream being processed and the one prefetched behind it
        self._last_slot = 1
        self._pending = []           # streams whose host->device copies are already queued (prefetch / run_many)
        self._dig = None
        self._host = None
        self._stage = [None, None]   # device blobs of the pieces in flight (double buffer)
        self.trace = None   # set to a list to collect (label, host ms since run() began) marks
        self.timing_hook = None   # called once per piece after its kernels are queued (bench: per-stage event spans)

    def schedule(self, n: int, ramp_up: bool = True):
        """Piece end offsets: sizes ramp x4 from piece/16 up to piece (unless the input is already arriving: a
        prefetched stream), and down again at the end."""
        lo = max(4 * self.cdc.max_size, (self.piece // 16) & ~15)
        up, s = [], lo
        while s < self.piece:
            up.append(s)
            s *= 4
        if n <= 2 * sum(up) + self.piece:   # short stream: equal pieces
            k = max(1, -(-n // self.piece))
            step = (-(-n // k) + 15) & ~15
            return [min(n, (i + 1) * step) for i in range(k)]
        ends, pos = [], 0
        for s in (up if ramp_up else []):
            pos += s
            ends.append(pos)
        tail = sum(up)
        while n - tail - pos > self.piece:
            pos += self.piece
            ends.append(pos)
        rest = n - tail - pos
        if rest > 0:
            pos += (rest + 15) & ~15 if rest % 16 and pos + ((rest + 15) & ~15) <= n - tail else rest & ~15
            if not ends or pos > ends[-1]:
                ends.append(pos)
        for s in reversed(up):
            pos = n if s == up[0] else min(n, pos + s)
            ends.append(pos)
        ends[-1] = n
        return [e for i, e in enumerate(ends) if i == 0 or e > ends[i - 1]]

    def _buffers(self, n: int, host_blob_cap: int):
        cap_chunks = n // self.cdc.min_size + 2
        if self._dig is None or self._dig.numel() < cap_chunks * 32:
            self._dig = self.ctx.empty(cap_chunks * 32, torch.uint8)
        h = self._host
        if h is None or h["cuts"].numel() < cap_chunks or h["blob"].numel() < host_blob_cap:
            h = self._host = {
                "cuts": torch.empty(cap_chunks, dtype=torch.int64, pin_memory=True),
                "digests": torch.empty(cap_chunks * 32, dtype=torch.uint8, pin_memory=True),
                "canon": torch.empty(cap_chunks, dtype=torch.int64, pin_memory=True),
                "offsets": torch.empty(cap_chunks + 1, dtype=torch.int64, pin_memory=True),
                "known": torch.empty(cap_chunks, dtype=torch.int64, pin_memory=True),
                "blob": torch.empty(host_blob_cap, dtype=torch.uint8, pin_memory=True)}
        return cap_chunks, h

    def _queue_in(self, host_in: torch.Tensor, ramp_up: bool = True):
        """Queues every host->device copy of one stream (piece by piece, an event per piece) on the copy stream, into
        the device input buffer that the previous stream does not occupy."""
        ctx = self.ctx
        n = host_in.numel()
        slot = self._last_slot ^ 1
        self._last_slot = slot
        if self._dbufs[slot] is None or self._dbufs[slot].numel() < n + 64:
            self._dbufs[slot] = None
            self._dbufs[slot] = ctx.empty(n + 64, torch.uint8)
        dbuf = self._dbufs[slot]
        ends = self.schedule(n, ramp_up) if n else [0]
        self.s_h2d.wait_stream(torch.cuda.current_stream(ctx.device))
        ev_in = []
        with torch.cuda.stream(self.s_h2d):
            a = 0
            for b in ends:
                if b > a:
                    dbuf[a:b].copy_(host_in[a:b], non_blocking=True)
                e = torch.cuda.Event()
                e.record(self.s_h2d)
                ev_in.append(e)
                a = b
        return {"key": (host_in.data_ptr(), n), "dbuf": dbuf, "ends": ends, "ev_in": ev_in}

    def prefetch(self, host_in: torch.Tensor, ramp_up: bool = False) -> None:
        """Starts copying the NEXT stream to the device behind the copies of the current one (at most one stream ahead):
        the following run(host_in) finds its input arriving or already there, so its piece schedule needs no ramp."""
        if len(self._pending) >= 2:
            raise RuntimeError("at most one stream can be prefetched ahead of the running one")
        self._pending.append(self._queue_in(host_in, ramp_up))

    def run_many(self, host_streams, host_blob_cap: Optional[int] = None, compress: bool = True):
        """A sequence of streams in pinned host memory: generator of HostIngestResult, each valid until the next is
        requested.  The input of stream k+1 is copied in while stream k is processed (its copies queue up behind
        stream k's), so only the first stream pays for the ramp of the piece schedule."""
        it = iter(host_streams)
        cur_h = next(it, None)
        if cur_h is None:
            return
        self.prefetch(cur_h, ramp_up=True)
        while cur_h is not None:
            nxt = next(it, None)
            if nxt is not None:
                self.prefetch(nxt)
            yield self.run(cur_h, host_blob_cap, compress)
            cur_h = nxt

    def run(self, host_in: torch.Tensor, host_blob_cap: Optional[int] = None, compress: bool = True,
            known=None) -> HostIngestResult:
        """known: as Ingest.run(known=...), piece by piece against the same archive (opened once per call); the result
        equals the run without it, plus `known` and `stats`."""
        import queue
        import threading
        import time
        ctx, cfg = self.ctx, self.cdc
        if host_in.is_cuda or host_in.dtype != torch.uint8 or host_in.dim() != 1:
            raise TypeError("host_in must be a 1-D uint8 host tensor (pinned for asynchronous copies)")
        n = host_in.numel()
        rd = self.open_known(known, compress) if known is not None else None
        stats = dict(copied=0, copied_bytes=0, compressed=0, compressed_raw_bytes=0) if known is not None else None
        t_run = time.perf_counter()

        def mark(label):
            if self.trace is not None:
                self.trace.append((label, (time.perf_counter() - t_run) * 1e3))
        if host_blob_cap is None:
            host_blob_cap = n + n // 64 + (1 << 20)
        cap_chunks, host = self._buffers(n, host_blob_cap)
        dig = self._dig
        cur = torch.cuda.current_stream(ctx.device)
        # every host->device copy is queued up front: the copy engine runs ahead of the kernels (already done when this
        # stream was prefetched)
        if self._pending and self._pending[0]["key"] == (host_in.data_ptr(), n):
            qin = self._pending.pop(0)
        else:
            if self._pending:
                raise RuntimeError("run() must be given the prefetched stream first")
            qin = self._queue_in(host_in)
        dbuf, ends, ev_in = qin["dbuf"], qin["ends"], qin["ev_in"]
        overlap = self.overlap and compress and len(ends) > 1
        mark("copies queued")
        host["offsets"][0] = 0

        def front(stream):
            """Pieces through scan, resolve, SHA-256, streaming dedup and selection, on `stream` with self.ctx."""
            ctx.check(ctx.lib.hmse_dedup_begin(ctx.h, cap_chunks, ctx.stream))
            entry = 0                  # absolute offset of the first chunk not yet cut
            n0 = 0                     # chunks before this piece
            for k, end in enumerate(ends):
                stream.wait_event(ev_in[k])
                eof = k == len(ends) - 1
                base = entry & ~15
                view = dbuf[base:end]
                n_own = end - base if eof else end - base - cfg.max_size
                if n_own <= entry - base:
                    continue           # (only when a piece is tiny) nothing can be decided yet
                mark("piece %d start" % k)
                ctx.chunk_scan(view, cfg)
                cuts, exit_off = ctx.chunk_resolve(view, cfg, n_own, eof, entry - base)
                mark("piece %d cuts" % k)
                nk = cuts.numel()
                if nk == 0:
                    continue
                dg = dig[n0 * 32:(n0 + nk) * 32]
                ctx.check(ctx.lib.hmse_digest(ctx.h, view.data_ptr(), entry - base, cuts.data_ptr(), nk, dg.data_ptr(),
                                              ctx.stream))
                canon = ctx.empty(nk, torch.int64)
                first = ctx.empty(nk, torch.uint8)
                ctx.check(ctx.lib.hmse_dedup_append(ctx.h, dig.data_ptr(), n0, nk, canon.data_ptr(), first.data_ptr(),
                                                    ctx.stream))
                sel = self.select_first(first) if compress else None
                cuts_abs = cuts + base
                mark("piece %d dedup" % k)
                ev = torch.cuda.Event()
                ev.record(stream)
                yield dict(k=k, view=view, start0=entry - base, cuts=cuts, cuts_abs=cuts_abs, nk=nk, n0=n0, dg=dg, canon=canon,
                           first=first, sel=sel, ev=ev)
                n0 += nk
                entry = base + exit_off

        if overlap:
            # the front stage of piece k+1 runs on its own thread, stream and hmse_ctx while piece k is compressed:
            # its kernels fill the gaps between the compression kernels, its host round trips cost nothing
            if self.ctx2 is None:
                self.ctx2 = Context(ctx.device)
                self.s_front = torch.cuda.Stream(ctx.tdev)
            self.s_front.wait_stream(cur)
            q: "queue.Queue" = queue.Queue(maxsize=2)
            stop = threading.Event()

            def put(item):
                while not stop.is_set():
                    try:
                        q.put(item, timeout=0.1)
                        return
                    except queue.Full:
                        pass

            def worker():
                try:
                    torch.cuda.set_device(ctx.device)
                    with torch.cuda.stream(self.s_front):
                        for rec in front(self.s_front):
                            put(rec)
                            if stop.is_set():
                                return
                    put(None)
                except BaseException as e:  # noqa: BLE001 - handed to the caller's thread
                    put(e)

            th = threading.Thread(target=worker, daemon=True)
            th.start()

            def records():
                while True:
                    item = q.get()
                    if item is None:
                        return
                    if isinstance(item, BaseException):
                        raise item
                    yield item
            back = self.ctx2
        else:
            stop, th = None, None
            records = lambda: front(cur)  # noqa: E731
            back = ctx

        keep = []                      # small device results stay referenced until the copies out have run
        ev_out = [None, None]          # copy-out of the piece that last used stage buffer j
        n_chunks = m_total = blob_total = 0
        d2h = 0
        try:
            for rec in records():
                k, nk = rec["k"], rec["nk"]
                cur.wait_event(rec["ev"])
                mk = bk = 0
                if compress:
                    j = k & 1
                    want = rec["view"].numel() // 2 + (1 << 20)
                    if self._stage[j] is None or self._stage[j].numel() < want:
                        self._stage[j] = None
                        self._stage[j] = back.empty(want, torch.uint8)
                    if ev_out[j] is not None:
                        cur.wait_event(ev_out[j])      # the buffer's previous contents have left the device
                    if known is not None:
                        blob, offs, kn, st = self.compress_known(rd, rec["view"], rec["cuts"], rec["dg"], rec["sel"],
                                                                 start0=rec["start0"], out=self._stage[j], ctx=back)
                        rec["known"] = kn
                        for key in stats:
                            stats[key] += st[key]
                    else:
                        blob, offs = back.compress(rec["view"], rec["cuts"], rec["sel"], self.zdict, self.level,
                                                   start0=rec["start0"], out=self._stage[j])
                    if blob.data_ptr() != self._stage[j].data_ptr():   # did not fit (poorly compressible): keep the larger one
                        self._stage[j] = blob
                    mk, bk = rec["sel"].numel(), blob.numel()
                    if blob_total + bk > host["blob"].numel():
                        raise ValueError("host_blob_cap %d is too small" % host["blob"].numel())
                    offs_abs = offs[1:] + blob_total
                    mark("piece %d compressed" % k)
                ev = torch.cuda.Event()
                ev.record(cur)
                self.s_d2h.wait_event(ev)
                with torch.cuda.stream(self.s_d2h):
                    host["cuts"][n_chunks:n_chunks + nk].copy_(rec["cuts_abs"], non_blocking=True)
                    host["digests"][n_chunks * 32:(n_chunks + nk) * 32].copy_(rec["dg"], non_blocking=True)
                    host["canon"][n_chunks:n_chunks + nk].copy_(rec["canon"], non_blocking=True)
                    d2h += nk * 48
                    if mk:
                        host["offsets"][1 + m_total:1 + m_total + mk].copy_(offs_abs, non_blocking=True)
                        host["blob"][blob_total:blob_total + bk].copy_(blob, non_blocking=True)
                        if known is not None:
                            host["known"][m_total:m_total + mk].copy_(rec["known"], non_blocking=True)
                        d2h += mk * 8 + bk
                        keep.append(offs_abs)
                        ev_out[k & 1] = torch.cuda.Event()
                        ev_out[k & 1].record(self.s_d2h)
                keep.append(rec)
                if self.timing_hook is not None and not overlap:
                    torch.cuda.current_stream(ctx.device).synchronize()
                    self.timing_hook()
                assert rec["n0"] == n_chunks
                n_chunks += nk
                m_total += mk
                blob_total += bk
        finally:
            if stop is not None:
                stop.set()
                th.join(timeout=30)
        mark("last piece queued")
        cur.wait_stream(self.s_d2h)    # the caller's stream (and its events) see the whole job
        if overlap:
            cur.wait_stream(self.s_front)
        torch.cuda.current_stream(ctx.device).synchronize()
        mark("done")
        del keep
        return HostIngestResult(host["cuts"][:n_chunks], host["digests"][:n_chunks * 32].view(n_chunks, 32),
                                host["canon"][:n_chunks], host["offsets"][:m_total + 1], host["blob"][:blob_total],
                                h2d_bytes=n, d2h_bytes=d2h, known=host["known"][:m_total] if known is not None else None,
                                stats=stats)


class CFabric:
    """The collectives of sharding.global_delta_bases served by the library (csrc/comm.cu) on ctx's own communicator."""

    def __init__(self, ctx: Context):
        self.ctx, self.world, self.rank = ctx, ctx.comm_world, ctx.comm_rank

    def allgather4(self, a, b=0, c=0, d=0):
        return self.ctx.allgather4(a, b, c, d)

    def lsh_exchange(self, keys):
        return self.ctx.lsh_exchange(keys)

    def alltoallv(self, send, send_counts, elem_bytes):
        return self.ctx.alltoallv(send, send_counts, elem_bytes)


class ShardedIngest(Ingest):
    """Rank r holds stream bytes [lo_r, hi_r + max_size) (the last rank up to the stream end).
    Chunks are owned by the shard they start in; global ids follow stream order."""

    def __init__(self, ctx: Context, cdc: CDCConfig = CDCConfig(), zdict=b"", level: int = 6, group=None,
                 transport: str = "auto"):
        """transport: "c" = the exchange steps run inside the library on its own NCCL communicator (hmse_chunk_sharded,
        hmse_dedup_global: one host round trip per step); "torch" = the same protocol spelled with torch.distributed
        collectives (hmse_b200/sharding.py - the form the gloo tests exercise on CPU); "auto" = "c" when the process
        group runs on NCCL."""
        super().__init__(ctx, cdc, zdict, level)
        self.group = group
        if transport == "auto":
            import torch.distributed as dist
            transport = "c" if dist.is_initialized() and dist.get_backend(group) == "nccl" else "torch"
        if transport not in ("c", "torch"):
            raise ValueError("transport must be 'auto', 'c' or 'torch'")
        self.transport = transport
        if transport == "c":
            ctx.comm_init(group)
        self._s_out = None
        self._s_in = None
        self._stage = [None, None]
        self._in = [None, None]
        self.trace = None      # set to a list: run_batches appends CUDA-event tuples per batch (bench.py's timeline)
        self.last_l4 = None

    def run(self, d: torch.Tensor, n_own: int, eof: bool, compress: bool = True, host=None, groups: int = 8,
            l4: Optional[SimConfig] = None, min_votes: int = 4):
        """One shard.  With `host` (pinned buffers from host_buffers()) the results are left in host memory and the
        compressed blob leaves the device in `groups` pieces while the rest is still being compressed.
        l4 (device results only): the similarity layer over the chunks that are first occurrences in the whole stream.
        With the C transport the LSH index is GLOBAL (similarity_delta_global): `base` holds global chunk ids and a base
        may live on another GPU - the result equals oracle.delta over the whole stream.  With the torch transport the
        layer runs shard-locally (`base` = local chunk indices; near duplicates whose original sits in another shard
        are stored whole).  Chunks that keep a delta are not compressed."""
        import torch.distributed as dist
        ctx = self.ctx
        dev = ctx.tdev
        world = dist.get_world_size(self.group)
        if self.transport == "c":
            cuts, entry, id_base, _ = ctx.chunk_sharded(d, self.cdc, n_own, eof)
            n = cuts.numel()
            digests = ctx.digest(d, cuts, start0=entry)
            canon, first = ctx.dedup_global(digests, id_base)
        else:
            ctx.chunk_scan(d, self.cdc)
            own = d.numel() if eof else n_own
            cuts, entry, _ = sharding.stitch_cuts(lambda e: ctx.chunk_resolve(d, self.cdc, n_own, eof, e), own, dev, self.group)
            n = cuts.numel()
            digests = ctx.digest(d, cuts, start0=entry)
            counts_all = sharding._all_gather_i64(n, dev, self.group)
            id_base = sum(counts_all[:dist.get_rank(self.group)])
            # partition -> all-to-all -> owner table -> all-to-all back -> scatter
            rec = ctx.empty(max(n, 1) * 40, torch.uint8)
            perm = ctx.empty(max(n, 1), torch.int32)
            cnt = (C.c_uint64 * world)()
            ctx.check(ctx.lib.hmse_dedup_partition(ctx.h, digests.data_ptr(), n, id_base, world, rec.data_ptr(), perm.data_ptr(),
                                                   cnt, ctx.stream))

            def owner(recv: torch.Tensor, m: int) -> torch.Tensor:
                out = ctx.empty(max(m, 1), torch.int64)
                ctx.check(ctx.lib.hmse_dedup_records(ctx.h, recv.data_ptr(), m, out.data_ptr(), ctx.stream))
                return out[:m]

            reply = sharding.exchange_dedup(rec[:n * 40], [int(c) for c in cnt], owner, self.group)
            canon = ctx.empty(max(n, 1), torch.int64)
            first = ctx.empty(max(n, 1), torch.uint8)
            ctx.check(ctx.lib.hmse_dedup_scatter(ctx.h, reply.data_ptr(), perm.data_ptr(), n, id_base, canon.data_ptr(),
                                                 first.data_ptr(), ctx.stream))
        canon, first = canon[:n], first[:n]
        base = dblob = doffs = None
        stored = first
        if l4 is not None and n:
            if host is not None:
                raise ValueError("l4 is not available together with host result buffers")
            if self.transport == "c":
                # global LSH index: bases may live on another GPU; `base` then holds GLOBAL chunk ids
                g = self.similarity_delta_global(d, cuts, first, entry, id_base, l4, min_votes)
                base, dblob, doffs = g["base_gid"], g["delta_blob"], g["delta_offsets"]
                self.last_l4 = g
            else:
                base, dblob, doffs = self.similarity_delta(d, cuts, first.view(torch.bool), l4, min_votes, start0=entry)
            stored = (first.view(torch.bool) & (base < 0)).view(torch.uint8)
        sel = self.select_first(stored)
        if host is not None:
            return self._compress_to_host(d, cuts, digests, canon, first, sel, entry, id_base, host, groups)
        if compress:
            blob, offs = ctx.compress(d, cuts, sel, self.zdict, self.level, start0=entry)
        else:
            blob, offs = ctx.empty(0, torch.uint8), ctx.empty(1, torch.int64).zero_()
        return IngestResult(cuts, digests, canon, first.view(torch.bool), sel, blob, offs, entry, id_base,
                            base=base, delta_blob=dblob, delta_offsets=doffs)

    def similarity_delta_global(self, d: torch.Tensor, cuts: torch.Tensor, first_u8: torch.Tensor, entry: int, id_base: int,
                                sim: SimConfig, min_votes: int = 4):
        """The L4 layer over the WHOLE stream (README.md:1553-1570: the LSH index a chunk probes is global): the chunks that
        are first occurrences anywhere are signed on their own rank, every band's keys go to the band's owner
        (hmse_lsh_exchange), the owners sort their bands and take the bucket heads (hmse_delta_heads), the heads travel
        back to the chunks' ranks, root flags are computed locally and gathered, bases are chosen among ALL roots, and the
        bytes of bases that live on another GPU are fetched (<= 32 KiB each) before the delta coding.  Equal to
        oracle.delta on the whole stream.  Returns a dict: base_gid int64[n] (GLOBAL chunk id of the base, -1 none),
        delta_blob, delta_offsets int64[n+1], plus what the read path needs (base_loc, ext_data, ext_off, ext_gid)."""
        ctx = self.ctx
        if not ctx.comm_world:
            raise RuntimeError("similarity_delta_global needs the C transport (ctx.comm_init)")
        dev = ctx.tdev
        n = cuts.numel()
        sel = self.select_first(first_u8)
        keys = ctx.lsh_keys(ctx.minhash(d, cuts, sim, start0=entry, select=sel), sim)            # [m, bands]
        starts = torch.cat([torch.full((1,), entry, dtype=torch.int64, device=dev), cuts[:-1]])
        lens = cuts - starts

        class Ops:
            @staticmethod
            def heads(owned):
                band, key, ids = ctx.lsh_buckets(owned.contiguous())
                return ctx.delta_heads(band, key, ids, int(owned.shape[0]), int(owned.shape[1]))

            @staticmethod
            def votes(heads, ubase, mv, root_all):
                return ctx.delta_votes(heads, ubase, mv, root_all=root_all)

            @staticmethod
            def chunk_bytes(want_j):
                lw = lens[want_j]
                out_off = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(lw, 0)])
                packed = ctx.empty(int(out_off[-1]) + 64, torch.uint8)
                if want_j.numel():
                    src_off = starts[want_j].contiguous()
                    ctx.check(ctx.lib.hmse_segment_copy(ctx.h, d.data_ptr(), src_off.data_ptr(), packed.data_ptr(),
                                                        out_off.data_ptr(), want_j.numel(), ctx.stream))
                return packed, lw

        g = sharding.global_delta_bases(CFabric(ctx), Ops, keys, sel, n, id_base, sim.bands, min_votes)
        base_loc, ext_off, ext_gid = g["base_loc"], g["ext_off"], g["ext_gid"]
        n_ext = int(ext_gid.numel())
        ext_store = ctx.empty(int(ext_off[-1]) + 64, torch.uint8)      # 8-byte aligned, slack behind the last base
        ext_store[:int(ext_off[-1])].copy_(g["ext_data"][:int(ext_off[-1])])
        dblob, doffs = ctx.delta_encode(d, cuts, base_loc, start0=entry, ext=(ext_store, ext_off) if n_ext else None)
        base_gid = torch.where(base_loc < 0, base_loc, torch.where(base_loc < n, base_loc + id_base,
                               ext_gid[(base_loc - n).clamp(min=0)] if n_ext else base_loc))
        return dict(base_gid=base_gid, delta_blob=dblob, delta_offsets=doffs, base_loc=base_loc, ext_data=ext_store, ext_off=ext_off,
                    ext_gid=ext_gid, n_remote=n_ext, n_unique=int(sel.numel()), exchange=ctx.exchange_stats())

    def run_batches(self, batches, n_own: int, eof: bool, host, groups: int = 8):
        """A sequence of shard buffers in pinned host memory (one per step of a continuous ingest): generator of
        HostIngestResult, one per batch, each valid until the next is requested.  The device input is double
        buffered - batch k+1 travels host->device on its own stream while batch k is chunked, deduplicated and
        compressed and its blob travels back - so a step costs max(copy in, compute, copy out) instead of their sum
        (global first-occurrence dedup needs every shard's digests before anything is compressed, so the copy in
        cannot be hidden inside one batch).  Every rank must iterate in step."""
        ctx = self.ctx
        cur = torch.cuda.current_stream(ctx.device)
        if self._s_in is None:
            self._s_in = torch.cuda.Stream(ctx.tdev)
        ready, free = [None, None], [None, None]
        marks = [None, None]      # (copy-in start, end) events of the batch in each slot, when tracing

        def fetch(slot: int, hb: torch.Tensor) -> int:
            n = hb.numel()
            if self._in[slot] is None or self._in[slot].numel() < n + 64:
                self._in[slot] = None
                self._in[slot] = ctx.empty(n + 64, torch.uint8)
            if free[slot] is not None:
                self._s_in.wait_event(free[slot])
            with torch.cuda.stream(self._s_in):
                if self.trace is not None:
                    t0 = torch.cuda.Event(enable_timing=True)
                    t0.record(self._s_in)
                self._in[slot][:n].copy_(hb.view(-1), non_blocking=True)
                ready[slot] = torch.cuda.Event(enable_timing=self.trace is not None)
                ready[slot].record(self._s_in)
                if self.trace is not None:
                    marks[slot] = (t0, ready[slot])
            return n

        it = iter(batches)
        nxt = next(it, None)
        if nxt is None:
            return
        n_cur, k = fetch(0, nxt), 0
        while True:
            slot = k & 1
            nxt = next(it, None)
            n_next = fetch(slot ^ 1, nxt) if nxt is not None else 0
            cur.wait_event(ready[slot])
            if self.trace is not None:
                c0 = torch.cuda.Event(enable_timing=True)
                c0.record(cur)
            res = self.run(self._in[slot][:n_cur], n_own, eof, host=host, groups=groups)
            free[slot] = torch.cuda.Event(enable_timing=self.trace is not None)
            free[slot].record(cur)
            if self.trace is not None:      # (copy-in start, copy-in end, pipeline start, everything incl. copy-out done)
                self.trace.append((marks[slot][0], marks[slot][1], c0, free[slot]))
            res.h2d_bytes = n_cur
            yield res
            if nxt is None:
                return
            n_cur, k = n_next, k + 1

    def host_buffers(self, n_avail: int):
        """Pinned result buffers for `run(..., host=...)`, sized for a shard buffer of n_avail bytes."""
        cap = n_avail // self.cdc.min_size + 2
        return {"cuts": torch.empty(cap, dtype=torch.int64, pin_memory=True),
                "digests": torch.empty(cap * 32, dtype=torch.uint8, pin_memory=True),
                "canon": torch.empty(cap, dtype=torch.int64, pin_memory=True),
                "offsets": torch.empty(cap + 1, dtype=torch.int64, pin_memory=True),
                "blob": torch.empty(n_avail // 2 + (1 << 20), dtype=torch.uint8, pin_memory=True)}

    def _compress_to_host(self, d, cuts, digests, canon, first, sel, entry, id_base, host, groups):
        """The selected chunks are compressed in `groups` runs; the blob of run g travels to the host while run g+1
        is compressed (two device buffers, a copy stream).  Streams and offsets equal one hmse_compress call."""
        ctx = self.ctx
        if self._s_out is None:
            self._s_out = torch.cuda.Stream(ctx.tdev)
        cur = torch.cuda.current_stream(ctx.device)
        n, m = cuts.numel(), sel.numel()
        ev0 = torch.cuda.Event()
        ev0.record(cur)
        self._s_out.wait_event(ev0)
        with torch.cuda.stream(self._s_out):
            host["cuts"][:n].copy_(cuts, non_blocking=True)
            host["digests"][:n * 32].copy_(digests.view(-1), non_blocking=True)
            host["canon"][:n].copy_(canon, non_blocking=True)
        host["offsets"][0] = 0
        d2h = n * 48
        per = max(1, -(-m // max(1, groups)))
        done = blob_total = 0
        ev_out = [None, None]
        keep = []
        g = 0
        while done < m:
            part = sel[done:done + per]
            j = g & 1
            want = d.numel() // (2 * max(1, groups)) + (8 << 20)
            if self._stage[j] is None or self._stage[j].numel() < want:
                self._stage[j] = None
                self._stage[j] = ctx.empty(want, torch.uint8)
            if ev_out[j] is not None:
                cur.wait_event(ev_out[j])
            blob, offs = ctx.compress(d, cuts, part, self.zdict, self.level, start0=entry, out=self._stage[j])
            if blob.data_ptr() != self._stage[j].data_ptr():
                self._stage[j] = blob
            mk, bk = part.numel(), blob.numel()
            if blob_total + bk > host["blob"].numel():
                raise ValueError("host blob buffer of %d bytes is too small" % host["blob"].numel())
            offs_abs = offs[1:] + blob_total
            ev = torch.cuda.Event()
            ev.record(cur)
            self._s_out.wait_event(ev)
            with torch.cuda.stream(self._s_out):
                host["offsets"][1 + done:1 + done + mk].copy_(offs_abs, non_blocking=True)
                host["blob"][blob_total:blob_total + bk].copy_(blob, non_blocking=True)
                ev_out[j] = torch.cuda.Event()
                ev_out[j].record(self._s_out)
            keep.append(offs_abs)
            d2h += mk * 8 + bk
            done += mk
            blob_total += bk
            g += 1
        cur.wait_stream(self._s_out)
        cur.synchronize()
        del keep
        res = HostIngestResult(host["cuts"][:n], host["digests"][:n * 32].view(n, 32), host["canon"][:n],
                               host["offsets"][:m + 1], host["blob"][:blob_total], h2d_bytes=0, d2h_bytes=d2h)
        res.entry, res.id_base = entry, id_base
        return res


class ShardedSimilarity:
    """MinHash / LSH over byte-range shards (BASELINE.json config 5): every rank signs its own chunks, the band
    keys travel to the band's owner (band % world) with one all-to-all, and the owner sorts its bands over ALL
    chunks of the stream - (band, key, global id) groups equal to oracle.buckets on the whole stream, band-sliced."""

    def __init__(self, ctx: Context, cfg=None, group=None, transport: str = "auto"):
        from .config import SimConfig
        self.ctx, self.cfg, self.group = ctx, cfg or SimConfig(), group
        if transport == "auto":
            import torch.distributed as dist
            transport = "c" if dist.is_initialized() and dist.get_backend(group) == "nccl" else "torch"
        self.transport = transport
        if transport == "c":
            ctx.comm_init(group)

    def run(self, d: torch.Tensor, cuts: torch.Tensor, start0: int = 0):
        """Returns (sig int32 [n, n_perm], keys int64 [n, bands], (band int32, key int64, id int64) of the owned bands)."""
        import torch.distributed as dist
        ctx = self.ctx
        sig = ctx.minhash(d, cuts, self.cfg, start0)
        keys = ctx.lsh_keys(sig, self.cfg)
        if self.transport == "c":
            owned, _ = ctx.lsh_exchange(keys)              # hmse_lsh_exchange: ncclSend / ncclRecv inside the library
            mine = list(range(owned.shape[1]))
        else:
            owned, mine, _ = sharding.exchange_lsh(keys, self.group)
        if owned.shape[0] == 0 or not mine:
            e32, e64 = ctx.empty(0, torch.int32), ctx.empty(0, torch.int64)
            return sig, keys, (e32, e64, e64.clone())
        band, key, ids = ctx.lsh_buckets(owned.contiguous())
        world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        band = band * world + rank          # local column -> global band number
        return sig, keys, (band, key, ids)


def verify_roundtrip(ctx: Context, res: IngestResult, zdict: torch.Tensor):
    """The read path over a whole ingest result, on the device: every compressed stream is inflated
    (hmse_inflate) and the SHA-256 of what comes out is compared with the digest taken from the source chunk at
    ingest.  Returns (streams that failed to inflate, all digests equal)."""
    sel = res.select
    m = sel.numel()
    if m == 0:
        return 0, True
    starts = torch.cat([torch.full((1,), res.entry, dtype=torch.int64, device=res.cuts.device), res.cuts[:-1]])
    lens = (res.cuts - starts)[sel]
    out_offs = torch.cat([torch.zeros(1, dtype=torch.int64, device=lens.device), torch.cumsum(lens, 0)])
    out, status, bad = ctx.inflate(res.blob, res.offsets, out_offs, zdict)
    dg = ctx.digest(out, out_offs[1:].contiguous())
    same = bool(torch.equal(dg, res.digests[sel]))
    return bad, same
