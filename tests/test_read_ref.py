"""CPU: the zlib-only range reader (tests/read_ref.py) on archives the oracle builds - v1, v2 (L4 deltas) and v3 (files):
its bytes equal slices of the input on random ranges, and it inflates exactly the stored chunks and delta bases the
ranges touch, counted independently with searchsorted over the pointer records."""
import numpy as np
import pytest

from oracle import corpus
from tests import read_ref


def _data(kind):
    base = corpus.generate(1 << 20)
    if kind == "v2":
        near = base[:512 << 10].copy()
        near[700::20000] ^= 0x20
        return np.concatenate([base, near, base[100 << 10:300 << 10]])
    return np.concatenate([base, base[200 << 10:400 << 10], base[:100 << 10]])


def _ranges(rng, raw, n, hi):
    ln = np.minimum(rng.integers(0, hi, n), raw)
    off = rng.integers(0, raw - ln + 1)
    return off, ln


@pytest.fixture(scope="module", params=["v1", "v2", "v3"])
def archive(request):
    kind = request.param
    data = _data(kind)
    sizes = None
    if kind == "v3":
        rng = np.random.default_rng(3)
        sizes = rng.integers(0, 24 << 10, 80)
        sizes[rng.random(80) < 0.2] = 0
        sizes[-1] = data.size - int(sizes[:-1].sum())
        assert sizes[-1] >= 0
    buf = read_ref.oracle_archive(data, corpus.zdict(), l4=kind == "v2", sizes=sizes)
    return kind, data, buf, sizes


def test_ranges_equal_input_slices(archive):
    kind, data, buf, _ = archive
    rng = np.random.default_rng(11)
    raw = data.size
    for hi in (2, 5000, 40000, 300000):
        off, ln = _ranges(rng, raw, 60, hi)
        st = {}
        got = read_ref.read(buf, off, ln, stats=st)
        assert got == [data[a:a + b].tobytes() for a, b in zip(off, ln)]
        slots, recs = read_ref.touched(buf, off, ln)
        assert st["inflated"] == slots.size and st["deltas"] == recs.size, (kind, hi, st, slots.size, recs.size)
    # whole stream, empty ranges (also at raw_bytes), one byte at the end
    assert read_ref.read(buf, [0, raw, 0, raw - 1], [raw, 0, 0, 1]) == [data.tobytes(), b"", b"", data[-1:].tobytes()]
    with pytest.raises(ValueError):
        read_ref.read(buf, [raw - 3], [4])


def test_v2_has_deltas_and_reads_touch_them(archive):
    kind, data, buf, _ = archive
    if kind != "v2":
        pytest.skip("deltas only in v2")
    slots, recs = read_ref.touched(buf, [0], [data.size])
    assert recs.size > 3
    st = {}
    read_ref.read(buf, [0], [data.size], stats=st)
    assert st["deltas"] == recs.size and st["inflated"] == slots.size


def test_file_relative_ranges(archive):
    kind, data, buf, sizes = archive
    if kind != "v3":
        pytest.skip("files only in v3")
    off = np.concatenate([[0], np.cumsum(sizes)])
    rng = np.random.default_rng(2)
    f = rng.integers(0, sizes.size, 50)
    ln = (rng.random(50) * (sizes[f] + 1)).astype(np.int64)
    a = (rng.random(50) * (sizes[f] - ln + 1)).astype(np.int64)
    got = read_ref.read(buf, a, ln, files=f)
    assert got == [data[off[x] + p:off[x] + p + q].tobytes() for x, p, q in zip(f, a, ln)]
    empty = int(np.flatnonzero(sizes == 0)[0])
    assert read_ref.read(buf, [0], [0], files=[empty]) == [b""]
    with pytest.raises(IndexError):
        read_ref.read(buf, [0], [0], files=[sizes.size])
    big = int(np.argmax(sizes))
    with pytest.raises(ValueError):
        read_ref.read(buf, [1], [int(sizes[big])], files=[big])
