"""CPU reference for composing archives (hmse_b200.archive.compose), numpy + zlib over container bytes (test
infrastructure).

compose(parts) takes (container bytes, files) pairs - files None for every file of the source (a v1 / v2 source is one
file), or a list of file indices of a v3 source - and returns the v3 container the rule of hmse_compose defines, walking
the output stream chunk by chunk in order:
  - one pointer record per output chunk, raw length copied from the source pointer;
  - a stored chunk is referenced directly or as the base of a referenced DeltaChunk record; its key is the output
    position of its first reference (a record's reference to its base counts at the record's chunk);
  - referenced stored chunks with equal digests are one chunk, the smaller key kept; kept chunks are numbered and their
    streams packed in key order;
  - a record, identified by (part, record position), is written once, numbered by first reference, base remapped;
  - refcounts: one per pointer on its slot and one per written record on its base, saturating at 65535.
Every part is a source of its own."""
from __future__ import annotations

import struct

import numpy as np

from oracle import archive as oarchive
from tests import files_ref


def _parse(buf: bytes):
    magic, ver, dlen, n, m, raw_bytes, sb, dad, n_delta, dsb = oarchive.HEADER.unpack_from(buf, 0)
    assert magic == oarchive.MAGIC and ver in (1, 2, 3)
    o = oarchive.HEADER.size
    zd = bytes(buf[o:o + dlen])
    o += dlen + ((-dlen) % 8)
    index = np.frombuffer(buf, dtype=np.uint8, count=m * 40, offset=o).reshape(m, 40)
    o += m * 40
    ptr = np.frombuffer(buf, dtype=np.uint8, count=n * 8, offset=o).reshape(n, 8)
    o += n * 8
    clen = index[:, 36:38].copy().view("<u2").reshape(-1).astype(np.int64)
    upos = np.concatenate([[0], np.cumsum(clen)]).astype(np.int64)
    pos = ptr[:, 0:4].copy().view("<u4").reshape(-1).astype(np.int64) * 512 + ptr[:, 4:6].copy().view("<u2").reshape(-1)
    raw = ptr[:, 6:8].copy().view("<u2").reshape(-1).astype(np.int64) + 1
    return dict(zd=zd, n=n, index=index, ptr=ptr, store=buf[o:o + sb], dstore=buf[o + sb:o + sb + dsb], sb=sb, upos=upos,
                pos=pos, raw=raw, slot=np.searchsorted(upos[:-1], np.minimum(pos, sb)), fc=files_ref.file_table(buf))


def compose(parts) -> bytes:
    src = [_parse(b) for b, _ in parts]
    zd = src[0]["zd"] if src else b""
    assert all(s["zd"] == zd for s in src), "the sources' dictionaries differ"
    stream, file_chunk = [], [0]   # (part, chunk) of every output chunk
    for p, ((_, files), s) in enumerate(zip(parts, src)):
        fc = s["fc"].astype(np.int64) if s["fc"] is not None else np.array([0, s["n"]], dtype=np.int64)
        if files is not None:
            assert s["fc"] is not None, "only v3 sources select files"
        for f in (range(fc.size - 1) if files is None else files):
            stream += [(p, i) for i in range(int(fc[f]), int(fc[f + 1]))]
            file_chunk.append(len(stream))
    # first references
    ukey, rkey, ref = {}, {}, []
    for q, (p, i) in enumerate(stream):
        s = src[p]
        if s["pos"][i] >= s["sb"]:
            dp = int(s["pos"][i]) - s["sb"]
            bslot = struct.unpack_from("<I", s["dstore"], dp)[0]
            rkey.setdefault((p, dp), q)
            ukey.setdefault((p, bslot), q)
            ref.append(("r", (p, dp)))
        else:
            ukey.setdefault((p, int(s["slot"][i])), q)
            ref.append(("u", (p, int(s["slot"][i]))))
    # stored chunks in key order, deduplicated by digest
    new_slot, kept, by_digest = {}, [], {}
    for key in sorted(ukey, key=ukey.get):
        p, k = key
        dg = src[p]["index"][k, :32].tobytes()
        if dg not in by_digest:
            by_digest[dg] = len(kept)
            kept.append(key)
        new_slot[key] = by_digest[dg]
    upos_out = np.concatenate([[0], np.cumsum([int(src[p]["index"][k, 36:38].view("<u2")[0]) for p, k in kept])]).astype(np.int64)
    store = b"".join(bytes(src[p]["store"][int(src[p]["upos"][k]):int(src[p]["upos"][k + 1])]) for p, k in kept)
    # records by first reference
    recs = sorted(rkey, key=rkey.get)
    rec_off, parts_d, off = {}, [], 0
    refcount = np.zeros(len(kept), dtype=np.int64)
    for p, dp in recs:
        ds = src[p]["dstore"]
        bslot, blen, dl = struct.unpack_from("<IHH", ds, dp)
        ns = new_slot[(p, bslot)]
        refcount[ns] += 1
        rec_off[(p, dp)] = off
        parts_d.append(struct.pack("<IHH", ns, blen, dl) + bytes(ds[dp + 8:dp + 8 + dl]))
        off += 8 + dl
    dstore = np.frombuffer(b"".join(parts_d), dtype=np.uint8)
    sb = len(store)
    ptr = np.zeros((len(stream), 8), dtype=np.uint8)
    for q, ((p, i), (kind, key)) in enumerate(zip(stream, ref)):
        if kind == "r":
            pos = sb + rec_off[key]
        else:
            ns = new_slot[key]
            pos = int(upos_out[ns])
            refcount[ns] += 1
        ptr[q, 0:4] = np.frombuffer(struct.pack("<I", pos >> 9), dtype=np.uint8)
        ptr[q, 4:6] = np.frombuffer(struct.pack("<H", pos & 511), dtype=np.uint8)
        ptr[q, 6:8] = src[p]["ptr"][i, 6:8]
    index = np.zeros((len(kept), 40), dtype=np.uint8)
    for ns, (p, k) in enumerate(kept):
        index[ns, :32] = src[p]["index"][k, :32]
        index[ns, 32:36] = np.frombuffer(struct.pack("<I", int(upos_out[ns]) >> 9), dtype=np.uint8)
        index[ns, 36:38] = src[p]["index"][k, 36:38]
        index[ns, 38:40] = np.frombuffer(struct.pack("<H", min(int(refcount[ns]), 0xFFFF)), dtype=np.uint8)
    raw_bytes = int(sum(int(src[p]["raw"][i]) for p, i in stream))
    return files_ref.pack(zd, index, ptr, np.frombuffer(store, dtype=np.uint8), raw_bytes, dstore, len(recs),
                          np.array(file_chunk, dtype=np.uint64))
