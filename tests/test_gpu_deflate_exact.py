"""GPU DEFLATE byte for byte: every stream hmse_compress writes must equal the stream of the sequential CPU model
(tests/model/deflate_model.cpp with the kernel's parameters: run heads with the kernel's sentinels before position 0,
2 / 3 / 4 own-chunk candidates by size class and 4 in every block of a long chunk, 4 dictionary candidates), or, for
stored streams, the one built in Python.  The inputs (tests/model/exact.py) cover what corpus text does not reach:
no, short and self-made dictionaries, the class boundaries at every staging alignment, binary and degenerate data
(P3b's CTA-wide sort, the 258 cap), multi-block chunks and their stored fallback, level 0, batch boundaries and the
dictionary cache.  A mismatch is reported with the first differing header field, code length or token."""
import time

import numpy as np
import pytest

from tests.model import exact
from tests.model.inflate_tokens import first_difference

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def model():
    return exact.Model()


def _run(ctx, case):
    import torch
    buf = ctx.empty(case.ptr_off + case.data.size + 64, torch.uint8)   # the allocator's blocks are 512-byte aligned
    d = buf[case.ptr_off:case.ptr_off + case.data.size]
    if case.data.size:
        d.copy_(torch.from_numpy(case.data))
    sel = None if case.select is None else ctx.stage_u64(case.select.astype(np.uint64))
    blob, offs = ctx.compress(d, ctx.stage_u64(case.cuts), sel, ctx.stage(case.zd), case.level, case.start0)
    return blob.cpu().numpy(), offs.cpu().numpy().view(np.uint64).astype(np.int64)


def _mismatches(case, blob, offs, expected, limit=5):
    if blob.tobytes() == b"".join(expected) and np.array_equal(np.diff(offs), [len(e) for e in expected]):
        return []
    assert offs.size == len(expected) + 1, "%s: %d offsets for %d streams" % (case.name, offs.size, len(expected))
    bad = []
    for k, (j, e) in enumerate(zip(case.order().tolist(), expected)):
        g = blob[offs[k]:offs[k + 1]].tobytes()
        if g != e:
            n = len(case.chunk(j))
            bad.append("%s: stream %d (chunk %d, %d bytes, %s class): gpu %d bytes, model %d bytes - %s" % (
                case.name, k, j, n, exact.size_class(n), len(g), len(e), first_difference(g, e)))
            if len(bad) >= limit:
                break
    return bad


@pytest.mark.parametrize("family", list(exact.FAMILIES))
def test_streams_equal_the_model(ctx, model, family):
    t0 = time.time()
    memo = {}
    bad, n_streams, n_distinct = [], 0, 0
    for case in exact.FAMILIES[family]():   # in order: the dictionary-cache family relies on consecutive calls
        blob, offs = _run(ctx, case)
        expected = case.expected(model, memo)
        n_streams += len(expected)
        n_distinct += len(set(case.order().tolist()))
        bad += _mismatches(case, blob, offs, expected)
    print("%s: %d streams (%d distinct chunks) equal the model, %.1f s" % (family, n_streams - len(bad), n_distinct,
                                                                           time.time() - t0))
    assert not bad, "%d stream(s) differ from the model:\n%s" % (len(bad), "\n".join(bad))


def test_block_count_limit(ctx, model):
    """A chunk of exactly 2048 blocks (64 MiB) is coded; one byte more is stored blocks, whatever the data."""
    n = 64 << 20
    zd = exact.zdict()
    data = np.zeros(n + 1, np.uint8)
    data[n // 2] = 1
    for length in (n, n + 1):
        case = exact.Case("blocks_%d" % length, data[:length], [length], zd)
        blob, offs = _run(ctx, case)
        want = exact.stored_stream(case.data, zd) if length > n else model.stream(case.data.tobytes(), zd)
        assert (length > n) == (len(want) > length), "the model's choice of block type is not the one under test"
        assert blob.tobytes() == want, "%d-byte chunk: %s" % (length, first_difference(blob.tobytes(), want))
