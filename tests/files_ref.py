"""CPU reference for many files in one call and the v3 archive container, built on the oracle (test infrastructure).

chunk_files runs the oracle's chunker on each file's bytes ALONE (the file is sliced out, its cuts shifted by its
offset), so that the GPU's single scan over the concatenated files is checked against a definition that does not
assume the locality it relies on.

Container v3 = v1 or v2 (oracle/archive.py) with version 3 and a file table behind the chunk store and the (possibly
empty) delta store: u64 n_files, u64 file_chunk[n_files + 1] (file f = chunks file_chunk[f] .. file_chunk[f+1]-1;
starts at 0, never decreases, ends at n_chunks).  restore(buf, files=[...]) walks only the pointer records of those
files and inflates, with zlib alone, only the stored chunks and delta bases they reference."""
from __future__ import annotations

import struct
import zlib

import numpy as np

from oracle import archive as oarchive
from oracle.cdc import _as_u8, chunk_c
from oracle.config import CDCConfig


def chunk_files(data, sizes, cfg: CDCConfig = CDCConfig(), impl=None):
    """Files held back to back in `data`, sizes[f] bytes each: (cuts uint64[n], file_chunk uint64[F+1]) with
    file_chunk[f] = index of file f's first chunk (an empty file shares its successor's), file_chunk[F] = n.
    impl(bytes, cfg) is the per-file chunker (default chunk_c)."""
    d = _as_u8(data)
    sizes = np.asarray(sizes, dtype=np.int64).reshape(-1)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    if (sizes < 0).any() or int(off[-1]) != d.size:
        raise ValueError("file sizes must be >= 0 and add up to len(data)")
    impl = impl or chunk_c
    parts, counts = [], []
    for f in range(sizes.size):
        c = np.asarray(impl(d[off[f]:off[f + 1]], cfg), dtype=np.uint64) + np.uint64(off[f])
        parts.append(c)
        counts.append(c.size)
    cuts = np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint64)
    file_chunk = np.concatenate([[0], np.cumsum(counts, dtype=np.int64)]).astype(np.uint64)
    return cuts.astype(np.uint64), file_chunk


def pack(zdict: bytes, index, pointers, store, raw_bytes: int, delta_store=None, n_delta: int = 0, file_chunk=None) -> bytes:
    """oracle.archive.pack, and with file_chunk the v3 container: version 3 and the file table appended."""
    buf = oarchive.pack(zdict, index, pointers, store, raw_bytes, delta_store, n_delta)
    if file_chunk is None:
        return buf
    fc = np.asarray(file_chunk, dtype=np.uint64)
    return buf[:8] + struct.pack("<I", 3) + buf[12:] + struct.pack("<Q", fc.size - 1) + fc.astype("<u8").tobytes()


def file_table(buf: bytes):
    """file_chunk uint64[n_files + 1] of a v3 container, None for v1 / v2; ValueError when the table is damaged."""
    magic, ver, dlen, n, m, raw_bytes, sb, dad, n_delta, dsb = oarchive.HEADER.unpack_from(buf, 0)
    if magic != oarchive.MAGIC or ver not in (1, 2, 3):
        raise ValueError("not an HMSE archive")
    if ver != 3:
        return None
    end = oarchive.HEADER.size + dlen + ((-dlen) % 8) + m * 40 + n * 8 + sb + dsb
    if end + 16 > len(buf):
        raise ValueError("archive size does not match its header")
    nf = struct.unpack_from("<Q", buf, end)[0]
    if end + 8 + 8 * (nf + 1) != len(buf):
        raise ValueError("file table size does not match the header")
    fc = np.frombuffer(buf, dtype="<u8", count=nf + 1, offset=end + 8).astype(np.uint64)
    if fc[0] != 0 or int(fc[-1]) != n or (np.diff(fc.astype(np.int64)) < 0).any():
        raise ValueError("file table must start at 0, never decrease and end at n_chunks")
    return fc


def restore(buf: bytes, files=None, stats=None):
    """Pure-Python read path of v1 / v2 / v3.  files (v3): a list of file indices; returns the list of those files'
    bytes, walking and inflating only what they reference.  `stats` (a dict) receives the number of zlib streams
    inflated ("inflated")."""
    from oracle.deltacode import delta_apply
    magic, ver, dlen, n, m, raw_bytes, sb, dad, n_delta, dsb = oarchive.HEADER.unpack_from(buf, 0)
    assert magic == oarchive.MAGIC and ver in (1, 2, 3)
    fc = file_table(buf) if files is not None else None
    assert files is None or fc is not None, "only v3 archives have a file table"
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
    lba = ptr[:, 0:4].copy().view("<u4").reshape(-1).astype(np.int64)
    off = ptr[:, 4:6].copy().view("<u2").reshape(-1).astype(np.int64)
    raw = ptr[:, 6:8].copy().view("<u2").reshape(-1).astype(np.int64) + 1
    pos = lba * 512 + off
    slot = np.searchsorted(upos, np.minimum(pos, sb))
    cache = {}

    def stored(s):
        if s not in cache:
            do = zlib.decompressobj(15, zd) if dlen else zlib.decompressobj(15)
            cache[s] = do.decompress(store[int(upos[s]):int(upos[s] + clen[s])]) + do.flush()
            assert do.eof
        return cache[s]

    def chunk(i):
        if pos[i] >= sb:   # DeltaChunk: read base -> inflate -> apply the delta
            dp = int(pos[i]) - sb
            bslot, blen, dl = struct.unpack_from("<IHH", dstore, dp)
            b = stored(bslot)
            assert len(b) == blen + 1
            return delta_apply(bytes(dstore[dp + 8:dp + 8 + dl]), b, int(raw[i]))
        s = int(slot[i])
        assert upos[s] == pos[i]
        assert len(stored(s)) == raw[i]
        return stored(s)

    def rebuild(rows):
        return b"".join(chunk(int(i)) for i in rows)

    if files is not None:
        out = [rebuild(range(int(fc[f]), int(fc[f + 1]))) for f in files]
    else:
        out = rebuild(range(n))
        assert len(out) == raw_bytes
    if stats is not None:
        stats["inflated"] = len(cache)
    return out
