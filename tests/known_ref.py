"""CPU reference for compressing against an opened archive (hmse_compress_known, Ingest.run(known=...)), numpy over
container bytes (test infrastructure).

known(buf, digests, lengths) gives, for every selected chunk (its SHA-256 and raw length), the archive slot whose zlib
stream is copied instead of compressing the chunk, or -1: the smallest slot whose index entry holds the chunk's digest,
when the stored chunk in that slot has the chunk's raw length.  A stored chunk's raw length comes from a pointer record
that addresses it, or from a DeltaChunk record whose base it is.  DeltaChunk targets have no index entry, so they are
never known."""
from __future__ import annotations

import struct

import numpy as np

from tests import compose_ref


def slot_lengths(buf: bytes):
    """(parsed container, raw length of every stored slot)."""
    p = compose_ref._parse(buf)
    ulen = np.full(p["index"].shape[0], -1, dtype=np.int64)
    direct = p["pos"] < p["sb"]
    ulen[p["slot"][direct]] = p["raw"][direct]
    for i in np.flatnonzero(~direct):
        base, blen1 = struct.unpack_from("<IH", p["dstore"], int(p["pos"][i]) - p["sb"])
        ulen[base] = blen1 + 1
    return p, ulen


def known(buf: bytes, digests, lengths) -> np.ndarray:
    p, ulen = slot_lengths(buf)
    first = {}
    for s in range(p["index"].shape[0]):
        first.setdefault(p["index"][s, :32].tobytes(), s)
    out = np.full(len(lengths), -1, dtype=np.int64)
    for k, (dg, ln) in enumerate(zip(digests, lengths)):
        s = first.get(bytes(np.asarray(dg, dtype=np.uint8)), -1)
        if s >= 0 and ulen[s] == int(ln):
            out[k] = s
    return out


def stream(buf: bytes, slot: int) -> bytes:
    """The zlib stream of a stored slot."""
    p = compose_ref._parse(buf)
    return bytes(p["store"][int(p["upos"][slot]):int(p["upos"][slot + 1])])
