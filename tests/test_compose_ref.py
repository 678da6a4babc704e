"""CPU: the compose reference (tests/compose_ref.py) on archives the oracle builds.  Composing archives of groups of files
gives the archive one ingest of the selected files, in order, gives - for merges, and for subsets with reorders and
repeats; composing one v3 archive alone is the identity, with or without deltas; with deltas every selected file reads
back; a delta's base whose own file was dropped is kept, ordered at the delta."""
import struct

import numpy as np
import pytest

from oracle import archive as oarchive
from oracle import corpus
from tests import compose_ref, files_ref, read_ref


def _files(seed, n, hi, data):
    rng = np.random.default_rng(seed)
    sizes = rng.integers(0, hi, n)
    sizes[rng.random(n) < 0.15] = 0
    sizes[-1] = 0
    sizes[-1] = data.size - int(sizes.sum())
    assert sizes[-1] >= 0
    return sizes


@pytest.fixture(scope="module")
def corpus_files():
    base = corpus.generate(1 << 20)
    data = np.concatenate([base[:600 << 10], base[100 << 10:300 << 10], base[:100 << 10]])
    sizes = _files(5, 60, 32 << 10, data)
    off = np.concatenate([[0], np.cumsum(sizes)])
    return data, sizes, [data[off[f]:off[f + 1]] for f in range(sizes.size)]


def _archive(files, l4=False):
    sizes = [f.size for f in files]
    data = np.concatenate(files) if files else np.zeros(0, dtype=np.uint8)
    return read_ref.oracle_archive(data, corpus.zdict(), l4=l4, sizes=sizes)


@pytest.mark.parametrize("groups", [2, 3])
def test_merge_equals_one_ingest(corpus_files, groups):
    data, sizes, files = corpus_files
    rng = np.random.default_rng(groups)
    cut = np.sort(rng.choice(np.arange(1, len(files)), groups - 1, replace=False))
    bounds = [0, *cut.tolist(), len(files)]
    parts = [(_archive(files[a:b]), None) for a, b in zip(bounds[:-1], bounds[1:])]
    assert compose_ref.compose(parts) == _archive(files)


def test_subset_with_reorder_and_repeats_equals_one_ingest(corpus_files):
    data, sizes, files = corpus_files
    a, b = _archive(files[:30]), _archive(files[30:])
    rng = np.random.default_rng(11)
    s1 = rng.integers(0, 30, 12).tolist() + [4, 4]
    s2 = rng.integers(0, len(files) - 30, 9).tolist()
    s3 = [7, 2, 7]
    parts = [(a, s1), (b, s2), (a, s3)]
    chosen = [files[f] for f in s1] + [files[30 + f] for f in s2] + [files[f] for f in s3]
    assert compose_ref.compose(parts) == _archive(chosen)


def test_v1_source_is_one_file(corpus_files):
    data, sizes, files = corpus_files
    v1 = read_ref.oracle_archive(data[:300 << 10], corpus.zdict())
    assert files_ref.file_table(v1) is None
    b = _archive(files[40:])
    whole = data[:300 << 10]
    assert compose_ref.compose([(v1, None), (b, None)]) == _archive([whole] + files[40:])


@pytest.fixture(scope="module")
def l4_files():
    base = corpus.generate(1 << 20)
    near = base[:512 << 10].copy()
    near[700::20000] ^= 0x20
    data = np.concatenate([base[:700 << 10], near, base[100 << 10:300 << 10]])
    sizes = _files(8, 40, 64 << 10, data)
    buf = read_ref.oracle_archive(data, corpus.zdict(), l4=True, sizes=sizes)
    n_delta = oarchive.HEADER.unpack_from(buf, 0)[8]
    assert n_delta > 10
    off = np.concatenate([[0], np.cumsum(sizes)])
    return buf, [data[off[f]:off[f + 1]].tobytes() for f in range(sizes.size)]


def test_identity(corpus_files, l4_files):
    buf = _archive(corpus_files[2])
    assert compose_ref.compose([(buf, None)]) == buf
    assert compose_ref.compose([(l4_files[0], None)]) == l4_files[0]


def test_deltas_restore(l4_files):
    buf, files = l4_files
    sel = [39, 3, 20, 20, 0, 35, 31]
    out = compose_ref.compose([(buf, sel[:4]), (buf, sel[4:])])
    assert oarchive.HEADER.unpack_from(out, 0)[8] > 0
    assert files_ref.restore(out, files=list(range(len(sel)))) == [files[f] for f in sel]


def _records(buf):
    p = compose_ref._parse(buf)
    recs = []
    for i in np.flatnonzero(p["pos"] >= p["sb"]):
        dp = int(p["pos"][i]) - p["sb"]
        recs.append((int(i), struct.unpack_from("<I", p["dstore"], dp)[0]))
    return p, recs


def test_base_of_a_dropped_file_is_kept_at_its_delta(l4_files):
    buf, files = l4_files
    p, recs = _records(buf)
    fc = p["fc"].astype(np.int64)
    file_of = np.searchsorted(fc, np.arange(p["n"]), side="right") - 1
    base_chunk = {int(p["slot"][i]): int(i) for i in np.flatnonzero(p["pos"] < p["sb"])[::-1]}
    i, bslot = next((i, b) for i, b in recs if file_of[base_chunk[b]] != file_of[i])
    f = int(file_of[i])
    out = compose_ref.compose([(buf, [f])])
    assert files_ref.restore(out, files=[0]) == [files[f]]
    q, _ = _records(out)
    dg = p["index"][bslot, :32].tobytes()
    digests = [q["index"][k, :32].tobytes() for k in range(q["index"].shape[0])]
    assert dg in digests
    # kept chunks are numbered by first reference: the base ranks after the stored chunks referenced before its delta
    j = i - int(fc[f])
    before = {int(q["slot"][c]) for c in range(j) if q["pos"][c] < q["sb"]}
    before |= {struct.unpack_from("<I", q["dstore"], int(q["pos"][c]) - q["sb"])[0] for c in range(j) if q["pos"][c] >= q["sb"]}
    if dg not in [digests[s] for s in before]:
        assert digests.index(dg) == len(before)
