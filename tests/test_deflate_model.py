"""The CPU side of the byte-exact DEFLATE tests: the token reader against stock zlib, the CPU model's streams against
stock zlib, the model's speed on degenerate input, and proof that the GPU test's inputs can tell the kernel's rules
from their neighbours (an input on which no rule change shows pins nothing).  No GPU needed."""
import ctypes as C
import time
import zlib

import numpy as np
import pytest

from tests.model import exact
from tests.model.inflate_tokens import first_difference, read_zlib, replay


@pytest.fixture(scope="module")
def model():
    return exact.Model()


def _inflate(stream, zd):
    d = zlib.decompressobj(zdict=zd) if zd else zlib.decompressobj()
    out = d.decompress(stream)
    assert d.eof and not d.unused_data, "not exactly one zlib stream"
    return out


# ---- the token reader ------------------------------------------------------------------------------------------

def _zlib_stream(data, level, strategy, zd):
    c = zlib.compressobj(level, zlib.DEFLATED, 15, 8, strategy, **({"zdict": zd} if zd else {}))
    return c.compress(data) + c.flush()


@pytest.mark.parametrize("level,strategy", [(0, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY),
                                            (6, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FIXED)])
@pytest.mark.parametrize("with_dict", [False, True])
def test_reader_replays_zlib_streams(level, strategy, with_dict):
    zd = exact.zdict() if with_dict else b""
    rng = np.random.default_rng(level)
    # text, a random stretch and text again: several blocks, stored ones among them at levels >= 1 too
    data = b"".join([exact.text(150000, 10).tobytes(), rng.integers(0, 256, 70000, dtype=np.uint8).tobytes(),
                     exact.text(50000, 3).tobytes(), bytes(300)])
    s = _zlib_stream(data, level, strategy, zd)
    st = read_zlib(s)
    assert st["end"] == len(s)
    assert st["dictid"] == (zlib.adler32(zd) if zd else None)
    assert st["adler"] == zlib.adler32(data)
    assert len(st["blocks"]) > 1 and st["blocks"][-1]["final"] and not any(b["final"] for b in st["blocks"][:-1])
    assert replay(st["blocks"], zd) == data
    types = {b["type"] for b in st["blocks"]}
    if level == 0:
        assert types == {0}
    elif strategy == zlib.Z_FIXED:   # fixed codes, stored blocks for the random stretch
        assert 1 in types and 2 not in types
    else:
        assert 2 in types
        if zd:   # the dictionary is used: some match reaches back before the first byte of the data
            pos, reach = 0, False
            for t in st["blocks"][0]["tokens"]:
                reach |= not isinstance(t, int) and t[1] > pos
                pos += 1 if isinstance(t, int) else t[0]
            assert reach


def test_first_difference_names_the_token(model):
    ch = exact.text(12000, 500).tobytes()
    a, b = model.stream(ch, exact.zdict()), model.stream(ch, exact.zdict(), own=1)
    assert first_difference(a, a) is None
    msg = first_difference(a, b)
    assert msg and "token" in msg, msg


# ---- the model -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("prev0", [0, 1])
@pytest.mark.parametrize("family", list(exact.FAMILIES))
def test_model_streams_inflate(model, family, prev0):
    n = 0
    for case in exact.FAMILIES[family]():
        sel = sorted(set(case.order().tolist()))
        chunks = [case.chunk(j) for j in sel]
        for ch, s in zip(chunks, model.streams(chunks, case.zd, case.level, prev0=prev0)):
            assert _inflate(s, case.zd) == ch, "%s: a %d-byte chunk does not round-trip" % (case.name, len(ch))
            assert len(s) <= len(ch) + 5 * (len(ch) // 65535 + 1) + 10
            n += 1
    assert n > 0


def test_long_stored_streams_equal_python(model):
    """The model's stored fallback and level 0 (multi-block chunks) are the streams built in Python; random data does
    not compress, so it takes the fallback."""
    rng = np.random.default_rng(4)
    for n in (32769, 65535, 65536, 2 * 65535, 200000):
        ch = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        for zd in (b"", exact.zdict()):
            want = exact.stored_stream(ch, zd)
            assert _inflate(want, zd) == ch
            assert model.stream(ch, zd) == want
            lib, pr = model.lib, exact.params(n)
            zdn = np.frombuffer(zd or b"\0", np.uint8)
            out = np.zeros(n + 1000, np.uint8)
            r = lib.model_compress_long(np.frombuffer(ch, np.uint8).ctypes.data, n, zdn.ctypes.data, len(zd), C.byref(pr), 0,
                                        out.ctypes.data, out.size)
            assert out[:r].tobytes() == want


def test_zeros_are_fast(model):
    """Runs used to cost the model quadratic time (every pair was extended to its end before the run-head test): only
    run heads are extended now."""
    for fill in (0, 0xFE):
        t0 = time.perf_counter()
        z = np.full(1 << 20, fill, np.uint8).tobytes()
        s = model.stream(z)
        s32 = model.stream(z[:32768])
        dt = time.perf_counter() - t0
        assert _inflate(s, b"") == z and _inflate(s32, b"") == z[:32768]
        assert dt < 5.0, "1 MiB of 0x%02x took %.1f s" % (fill, dt)


# ---- the GPU test's inputs can fail ----------------------------------------------------------------------------

def _differs(model, chunks, zd, **rule):
    """Number of chunks whose model stream changes when the kernel's rules are changed as given."""
    base = model.streams(chunks, zd)
    alt = model.streams(chunks, zd, **rule)
    return sum(a != b for a, b in zip(base, alt))


def test_each_sentinel_vector_pins_prev0(model):
    for name, ch, zd in exact.sentinel_vectors():
        assert _differs(model, [ch], zd, prev0=0) == 1, name
    for name, ch in exact.sentinel_long_vectors():
        for zd in (b"", exact.zdict()):
            assert _differs(model, [ch], zd, prev0=0) == 1, name


def _class_chunks(cls):
    """Chunks of one size class from the dictionary and length families of the GPU test, with their dictionaries."""
    out = []
    for case in exact.family_dicts()[:2] + exact.family_lengths()[:2] + exact.family_binary()[:4] + exact.family_long()[:1]:
        for j in range(case.cuts.size):
            ch = case.chunk(j)
            if exact.size_class(len(ch)) == cls:
                out.append((ch, case.zd))
    return out


@pytest.mark.parametrize("cls,own", [("small", 2), ("medium", 3), ("large", 4), ("long", 4)])
def test_inputs_pin_the_own_candidate_count(model, cls, own):
    chunks = _class_chunks(cls)
    assert chunks
    for zd in {z for _, z in chunks}:
        sub = [c for c, z in chunks if z == zd]
        assert exact.own_of(len(sub[0])) == own
        if _differs(model, sub, zd, own=own - 1):
            return
    pytest.fail("no %s-class chunk changes with %d instead of %d own candidates" % (cls, own - 1, own))


def test_inputs_pin_the_dictionary_cap(model):
    case = exact.family_dicts()[0]
    chunks = [case.chunk(j) for j in range(case.cuts.size)]
    assert _differs(model, chunks, case.zd, dict_cap=exact.DICT_CAP - 1) > 0


def test_dictionary_cache_inputs_tell_the_dictionaries_apart(model):
    """The dictionary-cache family compares a dictionary with one of the same length and Adler-32: the streams must
    differ, or a cache that confused the two would pass."""
    a, b, a2, _ = exact.dict_cache_dicts()
    case = exact.family_dict_cache()[0]
    chunks = [case.chunk(j) for j in range(case.cuts.size)]
    sa, sa2, sb = model.streams(chunks, a), model.streams(chunks, a2), model.streams(chunks, b)
    assert sa != sa2 and sa != sb and sa2 != sb
