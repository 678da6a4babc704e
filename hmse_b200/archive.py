"""The ingest result as a usable artefact: the spec's on-disk records (40-byte `ChunkIndex` entries,
README.md:1264-1269; 8-byte pointer records, README.md:1312; the packed chunk store, README.md:1879-1887) in one
container, written from the device results and read through the device read path (README.md:1617-1675): `Reader`
opens an archive once (hmse_read_open checks the records and derives the layout on the device) and serves batches of
byte ranges (hmse_read: every stored chunk and delta a batch needs is inflated / applied once, then the pieces are
copied out); `restore` is one range per stream or per file; `compose` turns files of several archives into one archive
on the device (hmse_compose: stored chunks deduplicated across sources by digest, streams and records copied, nothing
inflated).

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
single files and Reader.read(..., files=...) reads ranges inside them; both inflate only the stored chunks (and delta
bases) the ranges reference.
The v1 / v2 layout is restated for the tests in oracle/archive.py, v3 in tests/files_ref.py."""
from __future__ import annotations

import ctypes as C
import struct
import zlib
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _lib
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


class Reader:
    """An archive opened for random-access reads on the device (hmse_read_open / hmse_read).  The store, the delta
    store, the dictionary, the index and the pointer records are copied to the device once (and kept: `compose` reads
    them), the records are checked and the layout reads need is derived on the device; every `read` then serves a batch
    of byte ranges.  Raises
    ValueError on a damaged archive (the failed check is named)."""

    def __init__(self, ar: Archive, ctx: Optional[Context] = None):
        ctx = ctx or default_context()
        self.ctx, self.ar = ctx, ar
        self.n, self.m, self.raw_bytes = ar.n_chunks, ar.n_unique, int(ar.raw_bytes)
        self.n_delta = int(ar.n_delta) if ar.delta_store is not None else 0
        self.zd = ctx.stage(ar.zdict)
        self.store = ctx.stage(ar.store)
        self.dstore = ctx.stage(ar.delta_store) if self.n_delta else None
        self.index = ctx.stage(np.ascontiguousarray(ar.index).reshape(-1))
        self.pointers = ctx.stage(np.ascontiguousarray(ar.pointers).reshape(-1))
        lib = ctx.lib
        nbytes = int(lib.hmse_read_layout_bytes(self.n, self.m, self.n_delta))
        self.layout = ctx.empty(nbytes, torch.uint8)
        rc = lib.hmse_read_open(ctx.h, self.index.data_ptr(), self.m, self.pointers.data_ptr(), self.n, int(ar.store.size),
                                self.dstore.data_ptr() if self.n_delta else None, int(ar.delta_store.size) if self.n_delta else 0,
                                self.n_delta, self.raw_bytes, self.zd.data_ptr() if len(ar.zdict) else None, len(ar.zdict),
                                self.layout.data_ptr(), nbytes, ctx.stream)
        if rc == _lib.HMSE_E_INVAL:
            raise ValueError((lib.hmse_last_error(ctx.h) or b"").decode("utf-8", "replace"))
        ctx.check(rc)
        self.file_start = None    # raw offset of every file (v3), and the end of the stream
        if ar.file_chunk is not None:
            raw = ar.pointers[:, 6:8].copy().view("<u2").reshape(-1).astype(np.int64) + 1
            start = np.concatenate([[0], np.cumsum(raw)])
            self.file_start = start[ar.file_chunk.astype(np.int64)]

    def src(self) -> "_lib.ComposeSrc":
        """The descriptor hmse_compose and hmse_compress_known take for this archive."""
        d = _lib.ComposeSrc()
        d.d_layout, d.d_index, d.d_pointers = self.layout.data_ptr(), self.index.data_ptr(), self.pointers.data_ptr()
        d.d_store, d.d_delta_store = self.store.data_ptr(), self.dstore.data_ptr() if self.n_delta else None
        d.n, d.m, d.n_delta = self.n, self.m, self.n_delta
        return d

    def file_size(self, f) -> np.ndarray:
        return self.file_start[np.asarray(f) + 1] - self.file_start[np.asarray(f)]

    def read(self, offsets, lengths, files=None, device_out: bool = False, stats: Optional[dict] = None):
        """(data, off): the bytes of ranges [offsets[r], offsets[r] + lengths[r]) of the raw stream packed in request
        order, data[off[r]:off[r+1]] for range r (numpy, or CUDA tensors with device_out).  files (v3): a file index per
        range, offsets relative to the file, and every range must lie inside its file.  Raises IndexError for a bad
        file index, ValueError for a range outside its file or the stream and for a range that needs a damaged chunk.
        `stats` receives the streams inflated ("inflated"), the deltas applied ("deltas") and the raw bytes inflated
        ("inflated_bytes") - every stored chunk and delta the batch needs counts once."""
        ctx = self.ctx
        to_np = lambda x: np.asarray(x.cpu().numpy() if isinstance(x, torch.Tensor) else x).reshape(-1)  # noqa: E731
        off, ln = to_np(offsets), to_np(lengths)
        if off.shape != ln.shape:
            raise ValueError("offsets and lengths differ in size")
        if (off.size and off.dtype.kind == "i" and (off < 0).any()) or (ln.size and ln.dtype.kind == "i" and (ln < 0).any()):
            raise ValueError("negative offset or length")
        off, ln = off.astype(np.uint64), ln.astype(np.uint64)
        if files is not None:
            if self.file_start is None:
                raise ValueError("this archive has no file table (only v3 archives read by file)")
            f = to_np(files).astype(np.int64)
            if f.shape != off.shape:
                raise ValueError("files and offsets differ in size")
            nf = self.file_start.size - 1
            if ((f < 0) | (f >= nf)).any():
                raise IndexError("file index out of range (%d files)" % nf)
            size = self.file_size(f).astype(np.uint64)
            if ((ln > size) | (off > size - np.minimum(ln, size))).any():
                raise ValueError("a range runs past the end of its file")
            off = off + self.file_start[f].astype(np.uint64)
        R = off.size
        ends = np.concatenate([[np.uint64(0)], np.cumsum(ln, dtype=np.uint64)])
        total = int(ends[-1]) if R else 0
        if R and total < int(ln.max()):
            raise ValueError("the ranges add up to more than 2^64 bytes")
        ranges = ctx.stage_u64(np.stack([off, ln], axis=1).reshape(-1)) if R else ctx.empty(2, torch.int64)
        out = ctx.empty(total + 64, torch.uint8)
        out_off = ctx.empty(R + 1, torch.int64)
        status = ctx.empty(max(R, 1), torch.int32)
        got, bad, st4 = C.c_uint64(0), C.c_uint64(0), (C.c_uint64 * 4)()
        rc = ctx.lib.hmse_read(ctx.h, self.layout.data_ptr(), self.n, self.m, self.n_delta, self.store.data_ptr(),
                               self.dstore.data_ptr() if self.n_delta else None, self.zd.data_ptr() if self.zd.numel() else None,
                               int(self.zd.numel()), ranges.data_ptr(), R, out.data_ptr(), total, out_off.data_ptr(),
                               C.byref(got), status.data_ptr(), C.byref(bad), st4, ctx.stream)
        if rc == _lib.HMSE_E_INVAL:
            raise ValueError((ctx.lib.hmse_last_error(ctx.h) or b"").decode("utf-8", "replace"))
        ctx.check(rc)
        if bad.value:
            first = int(torch.nonzero(status[:R])[0])
            raise ValueError("%d ranges need a damaged chunk (first: range %d, status %d)" % (bad.value, first, int(status[first])))
        if stats is not None:
            stats.update(inflated=int(st4[0]), deltas=int(st4[1]), inflated_bytes=int(st4[2]))
        data = out[:total]
        if device_out:
            return data, out_off
        return data.cpu().numpy(), out_off.cpu().numpy().view(np.uint64)


def restore(ar: Archive, ctx: Optional[Context] = None, device_out: bool = False, files=None, stats: Optional[dict] = None):
    """The read path, through `Reader`: the stored chunks needed are inflated once each on the device, and the output is
    rebuilt from the pointer records.  files=None: returns the raw stream (numpy, or a CUDA tensor with device_out) - one
    range (0, raw_bytes).  files = a sequence of file indices (v3 archives): returns a list with the bytes of each
    requested file, in the order asked - one range per file, so only the stored chunks those files reference, and the
    bases of their deltas, are inflated.  `stats` (a dict) receives the number of zlib streams inflated ("inflated")
    and deltas applied ("deltas").  Raises ValueError on a damaged archive."""
    ctx = ctx or default_context()
    empty = lambda: ctx.empty(0, torch.uint8) if device_out else np.zeros(0, dtype=np.uint8)  # noqa: E731
    if files is not None:
        if ar.file_chunk is None:
            raise ValueError("this archive has no file table (only v3 archives restore single files)")
        fsel = np.asarray(files, dtype=np.int64).reshape(-1)
        if ((fsel < 0) | (fsel >= ar.n_files)).any():
            raise IndexError("file index out of range (%d files)" % ar.n_files)
    if stats is not None:
        stats.update(inflated=0, deltas=0)
    if ar.n_chunks == 0:
        return empty() if files is None else [empty() for _ in fsel]
    rd = Reader(ar, ctx)
    st = {}
    if files is None:
        data, _ = rd.read([0], [rd.raw_bytes], device_out=device_out, stats=st)
    else:
        data, off = rd.read(np.zeros(fsel.size, dtype=np.uint64), rd.file_size(fsel), files=fsel, device_out=device_out, stats=st)
        off = off.cpu().numpy().view(np.uint64) if isinstance(off, torch.Tensor) else off
    if stats is not None:
        stats.update(inflated=st["inflated"], deltas=st["deltas"])
    if files is None:
        return data
    return [data[int(a):int(b)] for a, b in zip(off[:-1], off[1:])]


def compose(parts, ctx: Optional[Context] = None, stats: Optional[dict] = None) -> Archive:
    """One v3 archive from files of several archives (hmse_compose): `parts` is a list of (source, files), a source an
    `Archive` (opened for this call) or a `Reader` (opened once, for many calls), files None for every file of the source
    (a v1 / v2 source is one file: its whole stream) or a list of file indices of a v3 source, in any order, repeats
    allowed.  File j of the result is the j-th file selected.  Stored chunks are numbered by first reference in the
    output stream and stored once per SHA-256 digest across sources, and their zlib streams and DeltaChunk records are
    copied without inflating anything: for sources without deltas the result is byte for byte the archive one
    `Ingest.run(files=...)` + `build` of the selected files, in that order, would write.  DeltaChunk records are not
    deduplicated across sources (the container stores no digest for them).  Every part is a source of its own, even
    when one archive appears in several parts.  `stats` receives "stored_referenced" (stored chunks referenced, before
    the digest dedup), "stored", "deduplicated", "records", "store_bytes" and "delta_store_bytes".  Raises ValueError
    for sources whose dictionaries differ, `files` on a source without a file table, an output of more than 2^32 - 2
    chunks (before any device work) or a store of 2 TiB or more, and IndexError for a file index out of range."""
    ctx = ctx or default_context()
    parts = list(parts)
    ars = [src.ar if isinstance(src, Reader) else src for src, _ in parts]
    zd = bytes(ars[0].zdict) if ars else b""
    if any(bytes(a.zdict) != zd for a in ars):
        raise ValueError("the sources' dictionaries differ")
    runs, sizes = [], []
    for p, (a, (_, files)) in enumerate(zip(ars, parts)):
        raw = a.pointers[:, 6:8].copy().view("<u2").reshape(-1).astype(np.int64) + 1
        cstart = np.concatenate([[0], np.cumsum(raw)])
        if files is None:
            fc = a.file_chunk.astype(np.int64) if a.file_chunk is not None else np.array([0, a.n_chunks], dtype=np.int64)
            f = np.arange(fc.size - 1)
        else:
            if a.file_chunk is None:
                raise ValueError("part %d: the source has no file table (only v3 sources select files)" % p)
            fc = a.file_chunk.astype(np.int64)
            f = np.asarray(files, dtype=np.int64).reshape(-1)
            if ((f < 0) | (f >= fc.size - 1)).any():
                raise IndexError("part %d: file index out of range (%d files)" % (p, fc.size - 1))
        first, cnt = fc[f], fc[f + 1] - fc[f]
        runs.append(np.stack([np.full(f.size, p), first, cnt], axis=1))
        sizes.append(cstart[fc[f + 1]] - cstart[first])
    runs = np.concatenate(runs) if runs else np.zeros((0, 3), dtype=np.int64)
    sizes = np.concatenate(sizes) if sizes else np.zeros(0, dtype=np.int64)
    file_chunk = np.concatenate([[0], np.cumsum(runs[:, 2])]).astype(np.uint64)
    n_out = int(file_chunk[-1])
    if n_out > 0xFFFFFFFE:
        raise ValueError("the output would hold %d chunks (at most 2^32 - 2)" % n_out)
    runs = runs[runs[:, 2] > 0]
    used = sorted(set(int(p) for p in runs[:, 0]))   # parts with chunks in the output: only these are opened
    empty = np.zeros((0, 40), dtype=np.uint8)
    if stats is not None:
        stats.update(stored_referenced=0, stored=0, deduplicated=0, records=0, store_bytes=0, delta_store_bytes=0)
    if n_out == 0:
        return Archive(zd, empty, np.zeros((0, 8), dtype=np.uint8), np.zeros(0, dtype=np.uint8), 0, None, 0, file_chunk)
    opened = {}
    for p in used:
        src = parts[p][0]
        if isinstance(src, Reader):
            opened.setdefault(id(src), src)
        elif id(src) not in opened:
            opened[id(src)] = Reader(src, ctx)
    readers = [opened[id(parts[p][0])] for p in used]
    slot = {p: k for k, p in enumerate(used)}
    runs[:, 0] = [slot[int(p)] for p in runs[:, 0]]
    descs = (_lib.ComposeSrc * len(readers))(*[rd.src() for rd in readers])
    sb = sum(int(rd.ar.store.size) for rd in readers)
    dsb = sum(int(rd.ar.delta_store.size) for rd in readers if rd.n_delta)
    icap = min(n_out, sum(rd.m for rd in readers))
    d_runs = ctx.stage_u64(runs.reshape(-1))
    ptrs = ctx.empty(8 * n_out, torch.uint8)
    index = ctx.empty(max(icap, 1) * 40, torch.uint8)
    store = ctx.empty(max(sb, 1), torch.uint8)
    dstore = ctx.empty(max(dsb, 1), torch.uint8)
    out6 = (C.c_uint64 * 6)()
    rc = ctx.lib.hmse_compose(ctx.h, descs, len(readers), d_runs.data_ptr(), runs.shape[0], n_out, ptrs.data_ptr(),
                              index.data_ptr(), icap, store.data_ptr(), sb, dstore.data_ptr(), dsb, out6, ctx.stream)
    if rc == _lib.HMSE_E_INVAL:
        raise ValueError((ctx.lib.hmse_last_error(ctx.h) or b"").decode("utf-8", "replace"))
    ctx.check(rc)
    _, cand, kept, sbytes, recs, dbytes = (int(x) for x in out6)
    if stats is not None:
        stats.update(stored_referenced=cand, stored=kept, deduplicated=cand - kept, records=recs, store_bytes=sbytes,
                     delta_store_bytes=dbytes)
    return Archive(zd, index[:kept * 40].cpu().numpy().reshape(kept, 40), ptrs.cpu().numpy().reshape(n_out, 8),
                   store[:sbytes].cpu().numpy(), int(sizes.sum()), dstore[:dbytes].cpu().numpy() if recs else None, recs,
                   file_chunk)
