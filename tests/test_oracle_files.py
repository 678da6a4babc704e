"""CPU: the per-file reference chunker (tests/files_ref.py, the oracle on each file alone) and the v3 archive container
with its file table."""
import struct

import numpy as np
import pytest

import oracle
from oracle import corpus
from oracle.config import CDCConfig as OCfg
from tests import files_ref

TINY = OCfg(64, 256, 1024, oracle.config.spread_mask(10), oracle.config.spread_mask(6))


def _sizes(rng, n_files, hi):
    s = rng.integers(0, hi, n_files)
    s[rng.random(n_files) < 0.2] = 0
    s[rng.random(n_files) < 0.1] = 1
    return s


@pytest.mark.parametrize("seed", range(6))
def test_chunk_files_equals_naive_per_file(seed):
    rng = np.random.default_rng(seed)
    sizes = _sizes(rng, int(rng.integers(1, 12)), 3000)
    data = corpus.generate(int(sizes.sum()) + 1)[:int(sizes.sum())] if seed % 2 else corpus.random_bytes(int(sizes.sum()), seed=seed)
    cuts, fc = files_ref.chunk_files(data, sizes, TINY)
    off = np.concatenate([[0], np.cumsum(sizes)])
    want, first = [], [0]
    for f in range(sizes.size):
        c = oracle.chunk_naive(data[off[f]:off[f + 1]], TINY) + np.uint64(off[f])
        want.append(c)
        first.append(first[-1] + c.size)
    assert np.array_equal(cuts, np.concatenate(want).astype(np.uint64))
    assert np.array_equal(fc, np.array(first, dtype=np.uint64))
    # every file ends with a cut, no chunk spans two files
    ends = off[1:][sizes > 0]
    assert np.isin(ends, cuts.astype(np.int64)).all()


def test_chunk_files_one_file_equals_chunk_c():
    d = corpus.generate(1 << 20)
    cuts, fc = files_ref.chunk_files(d, [d.size])
    assert np.array_equal(cuts, oracle.chunk_c(d))
    assert fc.tolist() == [0, cuts.size]


def test_chunk_files_empty_and_bad_sizes():
    cuts, fc = files_ref.chunk_files(np.zeros(0, np.uint8), [0, 0, 0])
    assert cuts.size == 0 and fc.tolist() == [0, 0, 0, 0]
    cuts, fc = files_ref.chunk_files(np.zeros(0, np.uint8), [])
    assert cuts.size == 0 and fc.tolist() == [0]
    with pytest.raises(ValueError):
        files_ref.chunk_files(np.zeros(10, np.uint8), [5, 4])
    with pytest.raises(ValueError):
        files_ref.chunk_files(np.zeros(10, np.uint8), [11, -1])


def _v3(data, sizes, zd=b""):
    cuts, fc = files_ref.chunk_files(data, sizes)
    dg = oracle.digest(data, cuts)
    canon, first = oracle.dedup(dg)
    sel = np.flatnonzero(first)
    blob, offs = oracle.compress(data, cuts, sel, zd)
    idx, ptr = oracle.archive.records(dg, canon, cuts, sel, offs)
    return files_ref.pack(zd, idx, ptr, blob, data.size, file_chunk=fc), fc, (idx, ptr, blob)


def test_v3_roundtrip_and_single_files():
    base = corpus.generate(600 << 10)
    sizes = np.array([100 << 10, 0, 1, 200 << 10, 100 << 10, 0, 0], dtype=np.int64)
    sizes[-1] = base.size - int(sizes[:-1].sum())
    data = base.copy()
    data[(300 << 10) + 1:(400 << 10) + 1] = data[:100 << 10]        # file 4 repeats file 0
    zd = corpus.zdict()
    buf, fc, (idx, ptr, blob) = _v3(data, sizes, zd)
    assert struct.unpack_from("<I", buf, 8)[0] == 3
    assert files_ref.file_table(buf).tolist() == fc.tolist()
    assert files_ref.restore(buf) == data.tobytes()
    off = np.concatenate([[0], np.cumsum(sizes)])
    st = {}
    got = files_ref.restore(buf, files=[4, 1, 2], stats=st)
    assert got == [data[off[f]:off[f + 1]].tobytes() for f in (4, 1, 2)]
    n4 = int(fc[5] - fc[4])
    assert 0 < st["inflated"] <= n4 + 1              # file 4's chunks and file 2's single byte, nothing else
    # without a file table the same records give the v1 container, byte for byte
    v1 = oracle.archive.pack(zd, idx, ptr, blob, data.size)
    assert struct.unpack_from("<I", v1, 8)[0] == 1 and buf[:8] == v1[:8] and buf[12:len(v1)] == v1[12:]
    assert len(buf) == len(v1) + 8 + 8 * fc.size


def test_v3_damage_is_rejected():
    data = corpus.generate(300 << 10)
    buf, fc, _ = _v3(data, [100 << 10, 0, 200 << 10])
    t = len(buf) - 8 * fc.size          # first entry of file_chunk
    n_chunks = int(fc[-1])

    def put(b, k, v):
        b = bytearray(b)
        struct.pack_into("<Q", b, t + 8 * k, v)
        return bytes(b)

    for bad in (put(buf, 0, 1),                               # does not start at 0
                put(buf, 2, int(fc[1]) - 1 if fc[1] else n_chunks + 5),   # decreases
                put(buf, 3, n_chunks - 1),                    # does not end at n_chunks
                buf[:-8],                                     # size disagrees with the header
                buf + b"\0" * 8,
                put(buf, -1, fc.size)):                       # n_files disagrees with the table's size
        with pytest.raises(ValueError):
            files_ref.file_table(bad)
