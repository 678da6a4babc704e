"""CPU: the known-chunk reference (tests/known_ref.py) on archives the oracle builds (v1, v2 with deltas, v3).  Every
known chunk's source stream inflates, with stock zlib and the dictionary, to that chunk's bytes; a chunk equal to a
DeltaChunk target is not known; a digest whose stored chunk has another raw length is not known."""
import zlib

import numpy as np
import pytest

import oracle
from oracle import corpus
from tests import compose_ref, files_ref, known_ref, read_ref


def _chunks(data, sizes=None):
    cuts = files_ref.chunk_files(data, sizes)[0] if sizes is not None else oracle.chunk_c(data)
    starts = np.concatenate([[0], cuts[:-1]]).astype(np.int64)
    return [data[int(a):int(b)] for a, b in zip(starts, cuts)]


def _lookup(buf, chunks):
    dg = [oracle.digest(c, np.array([c.size], dtype=np.uint64))[0] for c in chunks]
    return known_ref.known(buf, dg, [c.size for c in chunks])


@pytest.fixture(scope="module")
def snapshot():
    base = corpus.generate(1 << 20)
    new = np.concatenate([base[:400 << 10], base[300 << 10:500 << 10].copy(), corpus.generate(200 << 10, corpus.CorpusConfig(seed=9))])
    new[450 << 10:(450 << 10) + 4] ^= 0x5A
    return base, new


def _check_streams(buf, chunks, kn):
    zd = corpus.zdict()
    assert (kn >= 0).sum() > 10 and (kn < 0).sum() > 10
    for c, s in zip(chunks, kn):
        if s >= 0:
            d = zlib.decompressobj(zdict=zd)
            assert d.decompress(known_ref.stream(buf, int(s))) + d.flush() == c.tobytes()


def test_v1(snapshot):
    base, new = snapshot
    buf = read_ref.oracle_archive(base, corpus.zdict())
    chunks = _chunks(new)
    _check_streams(buf, chunks, _lookup(buf, chunks))


def test_v3(snapshot):
    base, new = snapshot
    rng = np.random.default_rng(3)
    sizes = rng.integers(0, 40 << 10, 30)
    sizes[-1] = base.size - int(sizes[:-1].sum())
    buf = read_ref.oracle_archive(base, corpus.zdict(), sizes=sizes)
    assert files_ref.file_table(buf) is not None
    chunks = _chunks(new, [new.size // 2, new.size - new.size // 2])
    _check_streams(buf, chunks, _lookup(buf, chunks))


def test_v2_delta_targets_are_not_known(snapshot):
    base, new = snapshot
    near = base[:512 << 10].copy()
    near[700::20000] ^= 0x20
    data = np.concatenate([base[:700 << 10], near])
    buf = read_ref.oracle_archive(data, corpus.zdict(), l4=True)
    p = compose_ref._parse(buf)
    targets = np.flatnonzero(p["pos"] >= p["sb"])
    assert targets.size > 10
    chunks = _chunks(data)
    assert (_lookup(buf, [chunks[i] for i in targets]) == -1).all()
    _check_streams(buf, _chunks(new), _lookup(buf, _chunks(new)))


def test_length_must_match(snapshot):
    base, new = snapshot
    buf = bytearray(read_ref.oracle_archive(base, corpus.zdict()))
    chunks = _chunks(new)
    kn = _lookup(bytes(buf), chunks)
    k = int(np.flatnonzero(kn < 0)[0])
    p, ulen = known_ref.slot_lengths(bytes(buf))
    s = int(np.flatnonzero(ulen != chunks[k].size)[0])
    off = bytes(buf).index(p["index"][s].tobytes())
    buf[off:off + 32] = oracle.digest(chunks[k], np.array([chunks[k].size], dtype=np.uint64))[0].tobytes()
    assert _lookup(bytes(buf), [chunks[k]])[0] == -1
