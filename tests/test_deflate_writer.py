"""The DEFLATE stream writer (tests/model/deflate_writer.py) and the decoder test's streams (tests/model/inflate_cases.py)
against stock zlib, no GPU needed: the writer is the exact inverse of the token reader on zlib's own streams, every
stream a family calls valid inflates under zlib to the bytes its tokens stand for, and zlib rejects every stream a
family calls invalid.  The GPU test trusts these labels only through zlib, so a wrong label fails here first."""
import zlib

import numpy as np
import pytest

from tests.model import deflate_writer as W
from tests.model import exact, inflate_cases
from tests.model.inflate_tokens import read_zlib


def _zlib_stream(data, level, strategy, zd):
    c = zlib.compressobj(level, zlib.DEFLATED, 15, 8, strategy, **({"zdict": zd} if zd else {}))
    return c.compress(data) + c.flush()


@pytest.mark.parametrize("level,strategy", [(0, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY),
                                            (6, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FIXED)])
@pytest.mark.parametrize("with_dict", [False, True])
def test_write_inverts_read_on_zlib_streams(level, strategy, with_dict):
    zd = exact.zdict() if with_dict else b""
    rng = np.random.default_rng(level + 10)
    data = b"".join([exact.text(150000, 20).tobytes(), rng.integers(0, 256, 70000, dtype=np.uint8).tobytes(),
                     exact.text(50000, 7).tobytes(), bytes(300)])
    for part in (data, data[:1], b""):
        s = _zlib_stream(part, level, strategy, zd)
        st = read_zlib(s)
        if part is data:
            assert len(st["blocks"]) > 1
        assert W.write_zlib(st) == s


def test_write_inverts_read_on_flushed_streams():
    """Sync and full flushes leave empty stored blocks and blocks that end mid-byte behind."""
    co = zlib.compressobj(6)
    d = exact.text(40000, 1).tobytes()
    s = co.compress(d[:10000]) + co.flush(zlib.Z_SYNC_FLUSH) + co.compress(d[10000:30000]) + \
        co.flush(zlib.Z_FULL_FLUSH) + co.compress(d[30000:]) + co.flush()
    st = read_zlib(s)
    assert any(b["type"] == 0 and not b["stored"] for b in st["blocks"])
    assert W.write_zlib(st) == s


def test_length_vector_helpers():
    for n, maxlen in [(286, 10), (286, 11), (286, 15), (30, 8), (30, 9), (30, 15), (16, 15), (13, 9)]:
        lens = W.spine_lens(n, maxlen)
        assert len(lens) == n and max(lens) == maxlen and lens.count(maxlen) == 2 and maxlen - 1 in lens
        assert W.kraft(lens) == 1 << 15
    for k in range(2, 300):
        assert W.kraft(W.balanced_lens(k)) == 1 << 15
    lens = [0] * 40
    lens[3] = 2
    W.fill_complete(lens, range(10, 40))
    assert W.kraft(lens) == 1 << 15


def _families():
    return {name: f() for name, f in inflate_cases.FAMILIES.items()}


@pytest.fixture(scope="module")
def families():
    return _families()


@pytest.mark.parametrize("family", list(inflate_cases.FAMILIES))
def test_family_labels_agree_with_zlib(families, family):
    n = {True: 0, False: 0, None: 0}
    bad = []
    for g in families[family]:
        names = [c.name for c in g.cases]
        assert len(set(names)) == len(names), "%s: case names repeat" % g.name
        for c in g.cases:
            got = inflate_cases.zlib_verdict(c.stream, g.zd, c.out_len)
            n[c.valid] += 1
            if c.valid is True and got != c.want:
                bad.append("%s / %s: zlib %s, expected %d bytes - %s" % (
                    g.name, c.name, "rejects it" if got is None else "gives other bytes", len(c.want),
                    inflate_cases.describe(c.stream)))
            if c.valid is False and got is not None:
                bad.append("%s / %s: zlib accepts a stream labelled invalid - %s" % (g.name, c.name,
                                                                                    inflate_cases.describe(c.stream)))
    assert not bad, "\n".join(bad)
    assert n[True] + n[False] + n[None] > 0
    if family == "damaged":   # three intact streams, every truncation and one flipped bit per byte of each
        assert n[True] == 3 and n[None] == 2 * sum(len(c.stream) for g in families[family] for c in g.cases if c.valid)


def test_valid_cases_read_back(families):
    """The writer's valid streams read back to the blocks they were written from (lengths, RLE, tokens)."""
    for g in families["code_shapes"] + families["dyn_headers"]:
        for c in (c for c in g.cases if c.valid):
            st = read_zlib(c.stream)
            assert st["end"] == len(c.stream), c.name
            assert W.write_zlib(st) == c.stream, c.name
