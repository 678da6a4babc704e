"""CPU reference for random-access reads of an archive (hmse_b200.archive.Reader.read), zlib only (test infrastructure).

read(buf, offsets, lengths, files=None) walks the container bytes of v1 / v2 / v3 (oracle/archive.py, tests/files_ref.py)
and returns the bytes of every range [offsets[r], offsets[r] + lengths[r]) of the raw stream; with files (v3) the
offsets are relative to the file and a range must lie inside it.  A stored chunk is inflated, and a DeltaChunk record
applied, only when a range touches it, once each; `stats` receives the streams inflated ("inflated"), the deltas
applied ("deltas") and the raw bytes inflated ("inflated_bytes"), as the device reader reports them."""
from __future__ import annotations

import struct
import zlib

import numpy as np

from oracle import archive as oarchive
from tests import files_ref


def read(buf: bytes, offsets, lengths, files=None, stats=None):
    from oracle.deltacode import delta_apply
    magic, ver, dlen, n, m, raw_bytes, sb, dad, n_delta, dsb = oarchive.HEADER.unpack_from(buf, 0)
    assert magic == oarchive.MAGIC and ver in (1, 2, 3)
    o = oarchive.HEADER.size
    zd = buf[o:o + dlen]
    o += dlen + ((-dlen) % 8)
    index = np.frombuffer(buf, dtype=np.uint8, count=m * 40, offset=o).reshape(m, 40)
    o += m * 40
    ptr = np.frombuffer(buf, dtype=np.uint8, count=n * 8, offset=o).reshape(n, 8)
    o += n * 8
    store = buf[o:o + sb]
    dstore = buf[o + sb:o + sb + dsb]
    clen = index[:, 36:38].copy().view("<u2").reshape(-1).astype(np.int64)
    upos = np.concatenate([[0], np.cumsum(clen)[:-1]])
    pos = ptr[:, 0:4].copy().view("<u4").reshape(-1).astype(np.int64) * 512 + ptr[:, 4:6].copy().view("<u2").reshape(-1)
    raw = ptr[:, 6:8].copy().view("<u2").reshape(-1).astype(np.int64) + 1
    chunk_off = np.concatenate([[0], np.cumsum(raw)])
    assert int(chunk_off[-1]) == raw_bytes
    slot = np.searchsorted(upos, np.minimum(pos, sb))
    offsets = [int(x) for x in np.asarray(offsets).reshape(-1)]
    lengths = [int(x) for x in np.asarray(lengths).reshape(-1)]
    if files is not None:
        fc = files_ref.file_table(buf)
        assert fc is not None, "only v3 archives have a file table"
        fstart = chunk_off[fc.astype(np.int64)]
        rel = []
        for f, a, ln in zip(np.asarray(files).reshape(-1), offsets, lengths):
            f = int(f)
            if not 0 <= f < fc.size - 1:
                raise IndexError("file index out of range")
            if a + ln > int(fstart[f + 1] - fstart[f]):
                raise ValueError("a range runs past the end of its file")
            rel.append(int(fstart[f]) + a)
        offsets = rel
    cache, dcache = {}, {}

    def stored(s):
        if s not in cache:
            do = zlib.decompressobj(15, zd) if dlen else zlib.decompressobj(15)
            cache[s] = do.decompress(store[int(upos[s]):int(upos[s] + clen[s])]) + do.flush()
            assert do.eof
        return cache[s]

    def chunk(i):
        if pos[i] >= sb:   # DeltaChunk: read base -> inflate -> apply the delta, once per record
            dp = int(pos[i]) - sb
            if dp not in dcache:
                bslot, blen, dl = struct.unpack_from("<IHH", dstore, dp)
                b = stored(bslot)
                assert len(b) == blen + 1
                dcache[dp] = delta_apply(bytes(dstore[dp + 8:dp + 8 + dl]), b, int(raw[i]))
            return dcache[dp]
        s = int(slot[i])
        assert upos[s] == pos[i]
        assert len(stored(s)) == raw[i]
        return stored(s)

    out = []
    for a, ln in zip(offsets, lengths):
        if a < 0 or ln < 0 or a + ln > raw_bytes:
            raise ValueError("a range runs past the end of the stream")
        parts = []
        if ln:
            c = int(np.searchsorted(chunk_off, a, side="right")) - 1
            while chunk_off[c] < a + ln:
                cs, ce = int(chunk_off[c]), int(chunk_off[c + 1])
                parts.append(chunk(c)[max(a, cs) - cs:min(a + ln, ce) - cs])
                c += 1
        out.append(b"".join(parts))
    if stats is not None:
        stats.update(inflated=len(cache), deltas=len(dcache), inflated_bytes=sum(len(v) for v in cache.values()))
    return out


def oracle_archive(data, zd: bytes = b"", l4: bool = False, sizes=None) -> bytes:
    """Container bytes of `data` built by the oracle alone: v1, v2 with l4 (near-duplicate chunks stored as deltas;
    v1 when none is kept), v3 with `sizes` (files chunked on their own)."""
    import oracle
    if sizes is not None:
        cuts, fc = files_ref.chunk_files(data, sizes)
    else:
        cuts, fc = oracle.chunk_c(data), None
    dg = oracle.digest(data, cuts)
    canon, first = oracle.dedup(dg)
    if l4:
        keys = oracle.band_keys(oracle.minhash_c(data, cuts))
        base, dblob, doffs = oracle.delta(data, cuts, keys, first)
        sel = np.flatnonzero(first & ~(base >= 0))
        blob, offs = oracle.compress(data, cuts, sel, zd)
        idx, ptr, dstore, nd = oarchive.records_l4(dg, canon, cuts, sel, offs, base, dblob, doffs)
        return files_ref.pack(zd, idx, ptr, blob, data.size, dstore, nd, fc)
    sel = np.flatnonzero(first)
    blob, offs = oracle.compress(data, cuts, sel, zd)
    idx, ptr = oarchive.records(dg, canon, cuts, sel, offs)
    return files_ref.pack(zd, idx, ptr, blob, data.size, file_chunk=fc)


def touched(buf: bytes, offsets, lengths):
    """(stored slots, DeltaChunk positions) the ranges need, counted with searchsorted over the pointer records alone:
    every chunk a non-empty range overlaps, its stored slot, or its record and the record's base slot."""
    magic, ver, dlen, n, m, raw_bytes, sb, dad, n_delta, dsb = oarchive.HEADER.unpack_from(buf, 0)
    o = oarchive.HEADER.size + dlen + ((-dlen) % 8)
    index = np.frombuffer(buf, dtype=np.uint8, count=m * 40, offset=o).reshape(m, 40)
    ptr = np.frombuffer(buf, dtype=np.uint8, count=n * 8, offset=o + m * 40).reshape(n, 8)
    dstore = np.frombuffer(buf, dtype=np.uint8, count=dsb, offset=o + m * 40 + n * 8 + sb)
    upos = np.concatenate([[0], np.cumsum(index[:, 36:38].copy().view("<u2").reshape(-1).astype(np.int64))[:-1]])
    pos = ptr[:, 0:4].copy().view("<u4").reshape(-1).astype(np.int64) * 512 + ptr[:, 4:6].copy().view("<u2").reshape(-1)
    ends = np.cumsum(ptr[:, 6:8].copy().view("<u2").reshape(-1).astype(np.int64) + 1)
    a = np.asarray(offsets, dtype=np.int64).reshape(-1)
    ln = np.asarray(lengths, dtype=np.int64).reshape(-1)
    a, ln = a[ln > 0], ln[ln > 0]
    c0 = np.searchsorted(ends, a, side="right")              # first chunk whose end lies past the first byte
    c1 = np.searchsorted(ends, a + ln - 1, side="right")     # the chunk that holds the last byte
    mark = np.zeros(n + 1, dtype=np.int64)
    np.add.at(mark, c0, 1)
    np.add.at(mark, c1 + 1, -1)
    rows = np.flatnonzero(np.cumsum(mark)[:n] > 0)
    p = pos[rows]
    recs = np.unique(p[p >= sb] - sb)
    bases = np.array([struct.unpack_from("<I", dstore, int(d))[0] for d in recs], dtype=np.int64)
    slots = np.unique(np.concatenate([np.searchsorted(upos, p[p < sb]), bases]).astype(np.int64))
    return slots, recs
