"""The ingest result as a usable artefact: the spec's on-disk records (40-byte `ChunkIndex` entries,
README.md:1264-1269; 8-byte pointer records, README.md:1312; the packed chunk store, README.md:1879-1887) in one
container, written from the device results and restored through the device read path (hmse_inflate +
hmse_segment_copy, README.md:1617-1675).

Container v1, little endian:
    0   magic b"HMSEARC1"
    8   u32 version (1), u32 dict_len
    16  u64 n_chunks, u64 n_unique, u64 raw_bytes, u64 store_bytes
    48  u32 dict_adler, 12 reserved bytes                                   (64-byte header)
    64  preset dictionary, zero padded to a multiple of 8
    ..  index:    n_unique x { sha256[32], u32 lba, u16 length, u16 refcount }   lba = store position >> 9
    ..  pointers: n_chunks x { u32 lba, u16 position & 511, u16 raw length - 1 }  (stream order)
    ..  store:    the zlib streams of the unique chunks, back to back
Limits of v1: chunks of 1..65536 bytes, compressed chunks below 64 KiB, stores below 2 TiB.
Container v2 (written only when the ingest ran the L4 layer and kept deltas) appends the delta store after the chunk
store: header bytes 52..55 = u32 n_delta, 56..63 = u64 delta_store_bytes; the delta store holds one `struct
DeltaChunk` (README.md:2182-2189) per kept delta: { u32 base = ChunkIndex entry number of the base chunk, u16 base raw
length - 1, u16 delta length, delta bytes (the COPY/ADD op list of hmse_delta_encode) }.  A pointer record whose
position lba * 512 + offset is >= store_bytes addresses the DeltaChunk at position - store_bytes; the read path inflates
the base, applies the delta (README.md:2191-2198) and checks nothing else - the digests of delta chunks are not stored.
Container v3 (written only when the ingest chunked files, `Ingest.run(files=...)`) is v1 or v2 with version 3 and a file
table after the chunk store and the delta store (which is empty, with n_delta == 0, when no deltas were kept):
    ..  u64 n_files, u64 file_chunk[n_files + 1]     file f = chunks file_chunk[f] .. file_chunk[f+1]-1 (stream order)
file_chunk starts at 0, never decreases and ends at n_chunks; an empty file has as many entries as any other.  The
table holds indices only: file names, modes and times are not part of the container.  restore(files=[...]) rebuilds
single files and inflates only the stored chunks (and delta bases) those files reference.
The v1 / v2 layout is restated for the tests in oracle/archive.py, v3 in tests/files_ref.py."""
from __future__ import annotations

import ctypes as C
import struct
import zlib
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from .api import Context, default_context

MAGIC = b"HMSEARC1"
HEADER = struct.Struct("<8sIIQQQQIIQ")


@dataclass
class Archive:
    zdict: bytes
    index: np.ndarray       # uint8 [n_unique, 40]
    pointers: np.ndarray    # uint8 [n_chunks, 8]
    store: np.ndarray       # uint8 [store_bytes]
    raw_bytes: int
    delta_store: Optional[np.ndarray] = None   # uint8: DeltaChunk records (container v2)
    n_delta: int = 0
    file_chunk: Optional[np.ndarray] = None    # uint64 [n_files + 1]: first chunk of every file (container v3)

    @property
    def n_chunks(self) -> int:
        return int(self.pointers.shape[0])

    @property
    def n_unique(self) -> int:
        return int(self.index.shape[0])

    @property
    def n_files(self) -> int:
        return int(self.file_chunk.size) - 1 if self.file_chunk is not None else 0

    def tobytes(self) -> bytes:
        pad = (-len(self.zdict)) % 8
        ds = self.delta_store if self.n_delta else None
        ver = 3 if self.file_chunk is not None else (2 if ds is not None else 1)
        hdr = HEADER.pack(MAGIC, ver, len(self.zdict), self.n_chunks, self.n_unique, self.raw_bytes,
                          int(self.store.size), zlib.adler32(self.zdict) if self.zdict else 0, self.n_delta if ds is not None else 0,
                          int(ds.size) if ds is not None else 0)
        ft = b""
        if self.file_chunk is not None:
            ft = struct.pack("<Q", self.n_files) + np.ascontiguousarray(self.file_chunk, dtype="<u8").tobytes()
        return b"".join([hdr, self.zdict, b"\0" * pad, self.index.tobytes(), self.pointers.tobytes(), self.store.tobytes(),
                         ds.tobytes() if ds is not None else b"", ft])

    def save(self, path: str) -> None:
        with open(path, "wb") as f:
            f.write(self.tobytes())

    @staticmethod
    def frombytes(buf) -> "Archive":
        mv = memoryview(buf)
        magic, ver, dlen, n, m, raw, sb, dad, n_delta, dsb = HEADER.unpack_from(mv, 0)
        if magic != MAGIC or ver not in (1, 2, 3) or (ver == 1 and (n_delta or dsb)) or (ver == 3 and dsb and not n_delta):
            raise ValueError("not an HMSE archive v1/v2/v3")
        o = HEADER.size
        zd = bytes(mv[o:o + dlen])
        if dlen and zlib.adler32(zd) != dad:
            raise ValueError("dictionary checksum mismatch")
        o += dlen + ((-dlen) % 8)
        index = np.frombuffer(mv, dtype=np.uint8, count=m * 40, offset=o).reshape(m, 40)
        o += m * 40
        pointers = np.frombuffer(mv, dtype=np.uint8, count=n * 8, offset=o).reshape(n, 8)
        o += n * 8
        store = np.frombuffer(mv, dtype=np.uint8, count=sb, offset=o)
        end = o + sb + dsb
        file_chunk = None
        if ver == 3:
            if end + 16 > len(mv):
                raise ValueError("archive size does not match its header")
            n_files = struct.unpack_from("<Q", mv, end)[0]
            if end + 8 + 8 * (n_files + 1) != len(mv):
                raise ValueError("file table size does not match the header")
            file_chunk = np.frombuffer(mv, dtype="<u8", count=n_files + 1, offset=end + 8).astype(np.uint64)
            if file_chunk[0] != 0 or int(file_chunk[-1]) != n or (np.diff(file_chunk.astype(np.int64)) < 0).any():
                raise ValueError("file table must start at 0, never decrease and end at n_chunks")
        elif end != len(mv):
            raise ValueError("archive size does not match its header")
        dstore = np.frombuffer(mv, dtype=np.uint8, count=dsb, offset=o + sb) if ver == 2 or (ver == 3 and n_delta) else None
        return Archive(zd, index, pointers, store, raw, dstore, n_delta, file_chunk)

    @staticmethod
    def load(path: str) -> "Archive":
        with open(path, "rb") as f:
            return Archive.frombytes(f.read())


def _dev(ctx: Context, t, dtype):
    if isinstance(t, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(t))
    t = t.contiguous()
    if t.dtype != dtype:
        t = t.view(dtype) if t.element_size() == torch.empty(0, dtype=dtype).element_size() else t.to(dtype)
    return t if t.is_cuda else t.to(ctx.tdev)


def build(res, zdict: bytes, raw_bytes: Optional[int] = None, ctx: Optional[Context] = None) -> Archive:
    """Archive of one ingest result (`IngestResult` on the device or `HostIngestResult`): index and pointer records
    are produced by hmse_index_build on the device.  A result with `file_chunk` (Ingest.run(files=...)) gives a v3
    container with its file table."""
    ctx = ctx or default_context()
    cuts = _dev(ctx, res.cuts, torch.int64)
    n = cuts.numel()
    digests = _dev(ctx, res.digests, torch.uint8).view(-1)
    canon = _dev(ctx, res.canon, torch.int64)
    sel = _dev(ctx, res.select, torch.int64)
    offs = _dev(ctx, res.offsets, torch.int64)
    m = sel.numel()
    entry = int(getattr(res, "entry", 0))
    id_base = int(getattr(res, "id_base", 0))
    index = ctx.empty(max(m, 1) * 40, torch.uint8)
    ptrs = ctx.empty(max(n, 1) * 8, torch.uint8)
    dstore, n_delta = None, 0
    base = getattr(res, "base", None)
    if base is not None and n:
        if id_base or entry:
            raise ValueError("archives with deltas are single-GPU (local chunk indices)")
        base = _dev(ctx, base, torch.int64)
        doffs = _dev(ctx, res.delta_offsets, torch.int64)
        dblob = _dev(ctx, res.delta_blob, torch.uint8)
        n_delta = int((base >= 0).sum())
        cap = int(doffs[-1]) + 8 * n_delta
        dbuf = ctx.empty(cap + 64, torch.uint8)
        got = C.c_uint64(0)
        ctx.check(ctx.lib.hmse_index_build_l4(ctx.h, digests.data_ptr(), canon.data_ptr(), cuts.data_ptr(), 0, n,
                                              sel.data_ptr(), m, offs.data_ptr(), base.data_ptr(), doffs.data_ptr(),
                                              dblob.data_ptr(), index.data_ptr(), ptrs.data_ptr(), dbuf.data_ptr(), cap,
                                              C.byref(got), ctx.stream))
        dstore = dbuf[:got.value].cpu().numpy()
    else:
        ctx.check(ctx.lib.hmse_index_build(ctx.h, digests.data_ptr(), canon.data_ptr(), id_base, cuts.data_ptr(), entry, n,
                                           sel.data_ptr(), m, offs.data_ptr(), index.data_ptr(), ptrs.data_ptr(), ctx.stream))
    blob = res.blob
    store = blob.cpu().numpy() if isinstance(blob, torch.Tensor) else np.asarray(blob)
    if raw_bytes is None:
        raw_bytes = (int(cuts[-1]) - entry) if n else 0
    fc = getattr(res, "file_chunk", None)
    if fc is not None:
        fc = (fc.cpu().numpy() if isinstance(fc, torch.Tensor) else np.asarray(fc)).astype(np.int64).astype(np.uint64)
    return Archive(bytes(zdict), index[:m * 40].cpu().numpy().reshape(m, 40), ptrs[:n * 8].cpu().numpy().reshape(n, 8),
                   np.ascontiguousarray(store), int(raw_bytes), dstore, n_delta, fc)


def restore(ar: Archive, ctx: Optional[Context] = None, device_out: bool = False, files=None, stats: Optional[dict] = None):
    """The read path: the stored chunks needed are inflated once each on the device, and the output is rebuilt from the
    pointer records.  files=None: returns the raw stream (numpy, or a CUDA tensor with device_out).  files = a sequence
    of file indices (v3 archives): returns a list with the bytes of each requested file, in the order asked; only the
    stored chunks those files reference, and the bases of their deltas, are gathered (hmse_segment_copy) and inflated.
    `stats` (a dict) receives the number of zlib streams inflated ("inflated") and deltas applied ("deltas").  Raises
    ValueError on a damaged archive."""
    ctx = ctx or default_context()
    n, m = ar.n_chunks, ar.n_unique
    empty = lambda: ctx.empty(0, torch.uint8) if device_out else np.zeros(0, dtype=np.uint8)  # noqa: E731
    if files is None:
        rows = None
    else:
        if ar.file_chunk is None:
            raise ValueError("this archive has no file table (only v3 archives restore single files)")
        fsel = np.asarray(files, dtype=np.int64).reshape(-1)
        if ((fsel < 0) | (fsel >= ar.n_files)).any():
            raise IndexError("file index out of range (%d files)" % ar.n_files)
        fc = ar.file_chunk.astype(np.int64)
        lo, cnt = fc[fsel], fc[fsel + 1] - fc[fsel]
        rows = np.repeat(lo - (np.cumsum(cnt) - cnt), cnt) + np.arange(int(cnt.sum()), dtype=np.int64)
    if stats is not None:
        stats.update(inflated=0, deltas=0)
    if n == 0:
        return empty() if files is None else [empty() for _ in fsel]
    idx = ar.index
    lba_u = idx[:, 32:36].copy().view(np.uint32).reshape(-1).astype(np.int64)
    clen = idx[:, 36:38].copy().view(np.uint16).reshape(-1).astype(np.int64)
    p = ar.pointers
    lba = p[:, 0:4].copy().view(np.uint32).reshape(-1).astype(np.int64)
    off = p[:, 4:6].copy().view(np.uint16).reshape(-1).astype(np.int64)
    raw = p[:, 6:8].copy().view(np.uint16).reshape(-1).astype(np.int64) + 1
    pos = lba * 512 + off
    is_delta = pos >= ar.store.size
    if is_delta.any() and (ar.delta_store is None or not ar.n_delta):
        raise ValueError("a pointer record addresses a delta store this archive does not have")
    dpos_all = pos - ar.store.size      # DeltaChunk position of the chunks stored as deltas
    pos = np.where(is_delta, 0, pos)    # (delta chunks are resolved below; slot 0 is a placeholder)
    # store positions of the index entries: sector from the entry, exact byte from the running sum of lengths
    upos = np.concatenate([[0], np.cumsum(clen)[:-1]])
    if not np.array_equal(upos >> 9, lba_u) or int(upos[-1] + clen[-1]) != ar.store.size:
        raise ValueError("index entries do not tile the chunk store")
    slot = np.searchsorted(upos, pos)
    if (slot >= m).any() or not np.array_equal(upos[slot], pos):
        raise ValueError("a pointer record does not address a stored chunk")
    # raw length of every unique chunk = raw length of any chunk pointing at it
    ulen = np.zeros(m, dtype=np.int64)
    ulen[slot[~is_delta]] = raw[~is_delta]
    dinfo = None
    rec = np.full(n, -1, dtype=np.int64)    # DeltaChunk record of every chunk stored as a delta
    if is_delta.any():
        # DeltaChunk headers: { u32 base slot, u16 base raw length - 1, u16 delta length }
        ds = ar.delta_store
        dpos, dinv = np.unique(dpos_all[is_delta], return_inverse=True)
        if (dpos < 0).any() or (dpos + 8 > ds.size).any():
            raise ValueError("a pointer record addresses outside the delta store")
        hdr = ds[(dpos[:, None] + np.arange(8)[None, :])]
        bslot = hdr[:, 0:4].copy().view("<u4").reshape(-1).astype(np.int64)
        blen = hdr[:, 4:6].copy().view("<u2").reshape(-1).astype(np.int64) + 1
        dlen = hdr[:, 6:8].copy().view("<u2").reshape(-1).astype(np.int64)
        if (bslot >= m).any() or (dpos + 8 + dlen > ds.size).any():
            raise ValueError("a DeltaChunk record is damaged")
        traw = np.zeros(dpos.size, dtype=np.int64)
        traw[dinv] = raw[is_delta]
        if not np.array_equal(traw[dinv], raw[is_delta]):
            raise ValueError("pointer records disagree about a delta chunk's length")
        known = ulen[bslot] != 0
        if not np.array_equal(ulen[bslot][known], blen[known]):
            raise ValueError("a DeltaChunk record disagrees with the pointer records about its base's length")
        ulen[bslot] = blen              # a base may be referenced by deltas only
        dinfo = (dpos, bslot, blen, dlen, traw)
        rec[is_delta] = dinv
    if (ulen == 0).any() or not np.array_equal(ulen[slot[~is_delta]], raw[~is_delta]):
        raise ValueError("pointer records disagree about a chunk's length")
    if int(raw.sum()) != ar.raw_bytes:
        raise ValueError("pointer records do not add up to the stream length")
    if rows is not None and rows.size == 0:
        return [empty() for _ in fsel]
    # what the requested chunks need: their stored chunks, their DeltaChunk records and those records' bases
    if rows is None:
        rows = np.arange(n, dtype=np.int64)
        need_r = np.arange(dinfo[0].size, dtype=np.int64) if dinfo is not None else np.zeros(0, dtype=np.int64)
        need_u = np.arange(m, dtype=np.int64)
    else:
        rd = is_delta[rows]
        need_r = np.unique(rec[rows[rd]])
        need_u = np.unique(np.concatenate([slot[rows[~rd]], dinfo[1][need_r] if dinfo is not None else []]).astype(np.int64))
    u_at = np.full(m, -1, dtype=np.int64)
    u_at[need_u] = np.arange(need_u.size)
    zd = ctx.stage(ar.zdict)
    store = ctx.stage(ar.store)
    if need_u.size == m:
        blob, offs = store, ctx.stage_u64(np.concatenate([upos, [ar.store.size]]).astype(np.uint64))
    else:
        # gather the streams of the needed chunks into one packed blob
        goff = np.concatenate([[0], np.cumsum(clen[need_u])]).astype(np.uint64)
        blob = ctx.empty(int(goff[-1]) + 64, torch.uint8)
        g_src, offs = ctx.stage_u64(upos[need_u].astype(np.uint64)), ctx.stage_u64(goff)   # named: they must outlive the call
        if need_u.size:
            ctx.check(ctx.lib.hmse_segment_copy(ctx.h, store.data_ptr(), g_src.data_ptr(), blob.data_ptr(), offs.data_ptr(),
                                                need_u.size, ctx.stream))
    uo = np.concatenate([[0], np.cumsum(ulen[need_u])]).astype(np.uint64)
    uniq, status, bad = ctx.inflate(blob, offs, ctx.stage_u64(uo), zd)
    if bad:
        raise ValueError("%d stored chunks failed to inflate (first: %d)" % (bad, int(need_u[int(torch.nonzero(status)[0])])))
    if stats is not None:
        stats.update(inflated=int(need_u.size), deltas=int(need_r.size))
    rows_d = is_delta[rows]
    src = np.zeros(rows.size, dtype=np.uint64)
    src[~rows_d] = uo[:-1][u_at[slot[rows[~rows_d]]]]
    if need_r.size:
        dpos, bslot, blen, dlen, traw = (x[need_r] for x in dinfo)
        r_at = np.full(dinfo[0].size, -1, dtype=np.int64)
        r_at[need_r] = np.arange(need_r.size)
        doff = np.concatenate([[0], np.cumsum(dlen)]).astype(np.uint64)
        dsd = ctx.stage(ar.delta_store)
        # gather the delta bytes of the records (they sit behind their 8-byte headers) into one packed blob
        dblob = ctx.empty(int(doff[-1]) + 64, torch.uint8)[:int(doff[-1])]
        t_src, t_dst = ctx.stage_u64((dpos + 8).astype(np.uint64)), ctx.stage_u64(doff)   # named: they must outlive the call
        ctx.check(ctx.lib.hmse_segment_copy(ctx.h, dsd.data_ptr(), t_src.data_ptr(), dblob.data_ptr(), t_dst.data_ptr(),
                                            dpos.size, ctx.stream))
        to = np.concatenate([[0], np.cumsum(traw)]).astype(np.uint64)
        bl = torch.from_numpy(blen.astype(np.uint32).view(np.int32).copy()).to(ctx.tdev)
        tout, dstatus, dbad = ctx.delta_apply(dblob, t_dst, uniq, ctx.stage_u64(uo[:-1][u_at[bslot]].astype(np.uint64)), bl,
                                              ctx.stage_u64(to))
        if dbad:
            raise ValueError("%d deltas failed to apply (first: %d)" % (dbad, int(torch.nonzero(dstatus)[0])))
        total_u = int(uo[-1])
        both = ctx.empty(total_u + int(to[-1]) + 64, torch.uint8)
        both[:total_u].copy_(uniq)
        both[total_u:total_u + int(to[-1])].copy_(tout)
        uniq = both
        src[rows_d] = np.uint64(total_u) + to[:-1][r_at[rec[rows[rows_d]]]]
    out_len = raw[rows]
    total = int(out_len.sum())
    out = ctx.empty(total + 64, torch.uint8)[:total]
    src_off = ctx.stage_u64(src)
    dst = np.concatenate([[0], np.cumsum(out_len)]).astype(np.uint64)
    dst_off = ctx.stage_u64(dst)
    if rows.size:
        ctx.check(ctx.lib.hmse_segment_copy(ctx.h, uniq.data_ptr(), src_off.data_ptr(), out.data_ptr(), dst_off.data_ptr(),
                                            rows.size, ctx.stream))
    if files is None:
        return out if device_out else out.cpu().numpy()
    res = out if device_out else out.cpu().numpy()
    ends = dst[np.cumsum(cnt)].astype(np.int64)
    return [res[int(a):int(b)] for a, b in zip(np.concatenate([[0], ends[:-1]]), ends)]
