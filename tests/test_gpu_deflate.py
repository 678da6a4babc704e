"""GPU parity: per-chunk preset-dictionary DEFLATE.  Streams are judged the way SURVEY.md §8b
says: every slice must be exactly one zlib stream that inflates (stock zlib, zdict) to the raw
chunk, and the total size must be within 2 % of zlib level 6.  Byte-for-byte equality with the
encoder's own CPU model is tests/test_gpu_deflate_exact.py."""
import zlib

import numpy as np
import pytest

import oracle
from oracle import corpus

pytestmark = pytest.mark.gpu


def _roundtrip(data, cuts, select, zd, blob, offs):
    assert offs.size == (len(select) if select is not None else cuts.size) + 1
    assert int(offs[0]) == 0 and int(offs[-1]) == blob.size
    outs = oracle.inflate_all(blob, offs, zd)
    starts = np.concatenate([[0], cuts[:-1]]).astype(np.int64)
    sel = np.arange(cuts.size) if select is None else np.asarray(select)
    raw = memoryview(np.ascontiguousarray(data))
    for k, j in enumerate(sel):
        want = bytes(raw[int(starts[j]):int(cuts[j])])
        assert outs[k] == want, "chunk %d (len %d) did not round-trip" % (j, len(want))


def _ratio_vs_zlib(data, cuts, select, zd, blob):
    zb, _ = oracle.compress(data, cuts, np.arange(cuts.size) if select is None else select, zd)
    return zb.size / blob.size


def test_corpus_chunks_with_dict(ctx, corpus8):
    import hmse_b200
    d = corpus8[:4 << 20]
    cuts = oracle.chunk_c(d)
    zd = corpus.zdict()
    blob, offs = hmse_b200.compress(d, cuts, None, zd, ctx=ctx)
    _roundtrip(d, cuts, None, zd, blob, offs)
    r = _ratio_vs_zlib(d, cuts, None, zd, blob)
    print("zlib6/gpu bytes = %.4f, ratio %.3f" % (r, d.size / blob.size))
    assert r >= 0.98


def test_corpus_unique_selection(ctx, corpus8):
    import hmse_b200
    d = corpus8
    cuts = oracle.chunk_c(d)
    _, first = oracle.dedup(oracle.digest(d, cuts))
    sel = np.flatnonzero(first)
    zd = corpus.zdict()
    blob, offs = hmse_b200.compress(d, cuts, sel, zd, ctx=ctx)
    _roundtrip(d, cuts, sel, zd, blob, offs)
    assert _ratio_vs_zlib(d, cuts, sel, zd, blob) >= 0.98


def test_no_dict(ctx, corpus8):
    import hmse_b200
    d = corpus8[:2 << 20]
    cuts = oracle.chunk_c(d)
    blob, offs = hmse_b200.compress(d, cuts, None, b"", ctx=ctx)
    _roundtrip(d, cuts, None, b"", blob, offs)
    assert blob[0] == 0x78 and blob[1] == 0x9C
    assert _ratio_vs_zlib(d, cuts, None, b"", blob) >= 0.98


@pytest.mark.parametrize("kib", [4, 8, 16, 32])
def test_fixed_size_chunks(ctx, corpus8, kib):
    # BASELINE.json config 3: fixed-size chunk sets, ratio vs zlib level 6 and round trip
    import hmse_b200
    d = corpus8[:4 << 20]
    sz = kib << 10
    cuts = np.arange(sz, d.size + 1, sz, dtype=np.uint64)
    zd = corpus.zdict()
    blob, offs = hmse_b200.compress(d, cuts, None, zd, ctx=ctx)
    _roundtrip(d, cuts, None, zd, blob, offs)
    r = _ratio_vs_zlib(d, cuts, None, zd, blob)
    print("%d KiB: zlib6/gpu bytes = %.4f" % (kib, r))
    assert r >= 0.98


def test_64k_chunks_ratio_and_roundtrip(ctx, corpus8):
    # BASELINE.json config 3, 64 KiB row: chunks longer than 32 KiB become multi-block streams whose blocks
    # see the previous 32 KiB (zlib's window), so the ratio bar holds there too
    import hmse_b200
    d = corpus8[:4 << 20]
    cuts = np.arange(65536, d.size + 1, 65536, dtype=np.uint64)
    zd = corpus.zdict()
    blob, offs = hmse_b200.compress(d, cuts, None, zd, ctx=ctx)
    _roundtrip(d, cuts, None, zd, blob, offs)
    r = _ratio_vs_zlib(d, cuts, None, zd, blob)
    print("64 KiB: zlib6/gpu bytes = %.4f" % r)
    assert r >= 0.98


def test_long_chunks_mixed(ctx, corpus8):
    # ragged long chunks (block edges at 32 KiB multiples +-1, a 1 MiB chunk, > 96 blocks in one call so that
    # several batches run), mixed with short ones, with and without a dictionary, level 0, incompressible
    import hmse_b200
    rng = np.random.default_rng(3)
    lens = [32769, 65535, 65536, 65537, 98304, 100, 40000, 1 << 20, 8192, 3 * 32768 + 5, 200000] + [70000] * 60
    d = corpus8[:sum(lens)].copy()
    d[300000:300000 + 150000] = rng.integers(0, 256, 150000, dtype=np.uint8)   # incompressible stretch
    cuts = np.cumsum(lens).astype(np.uint64)
    zd = corpus.zdict()
    for z in (zd, b""):
        blob, offs = hmse_b200.compress(d, cuts, None, z, ctx=ctx)
        _roundtrip(d, cuts, None, z, blob, offs)
        assert _ratio_vs_zlib(d, cuts, None, z, blob) >= 0.975
        blob2, offs2 = hmse_b200.compress(d, cuts, None, z, ctx=ctx)
        assert np.array_equal(blob, blob2) and np.array_equal(offs, offs2)      # deterministic
    blob0, offs0 = hmse_b200.compress(d, cuts, None, zd, level=0, ctx=ctx)
    _roundtrip(d, cuts, None, zd, blob0, offs0)
    sizes = np.diff(offs.astype(np.int64))
    assert (sizes <= np.array([hmse_b200.compress_bound(int(n)) for n in lens])).all()
    r = rng.integers(0, 256, 200000, dtype=np.uint8)
    rc = np.array([70000, 200000], dtype=np.uint64)
    blob, offs = hmse_b200.compress(r, rc, None, zd, ctx=ctx)
    _roundtrip(r, rc, None, zd, blob, offs)
    assert blob.size <= r.size + 64


def test_header_bytes_and_dictid(ctx, corpus8):
    import hmse_b200
    d = corpus8[:100000]
    cuts = oracle.chunk_c(d)
    zd = corpus.zdict()
    blob, offs = hmse_b200.compress(d, cuts, None, zd, ctx=ctx)
    for a in offs[:-1].tolist():
        assert blob[a] == 0x78 and blob[a + 1] == 0xBB          # CMF/FLG with FDICT (SURVEY.md §4)
        assert int.from_bytes(bytes(blob[a + 2:a + 6]), "big") == zlib.adler32(zd)


def test_incompressible_falls_back_to_stored(ctx):
    # VALIDATION_METHODS.md:213 control corpus: CF 1.0, must still round-trip
    import hmse_b200
    d = corpus.random_bytes(1 << 20)
    cuts = oracle.chunk_c(d)
    blob, offs = hmse_b200.compress(d, cuts, None, corpus.zdict(), ctx=ctx)
    _roundtrip(d, cuts, None, corpus.zdict(), blob, offs)
    assert blob.size <= d.size + 16 * cuts.size


@pytest.mark.parametrize("fill", [0, 0x41])
def test_constant_chunks(ctx, fill):
    import hmse_b200
    d = np.full(300000, fill, dtype=np.uint8)
    cuts = oracle.chunk_c(d)
    blob, offs = hmse_b200.compress(d, cuts, None, b"", ctx=ctx)
    _roundtrip(d, cuts, None, b"", blob, offs)
    assert blob.size < d.size // 50


def test_tiny_and_ragged_chunks(ctx, corpus8):
    import hmse_b200
    lens = np.array([0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 100, 257, 258, 259, 260, 1000,
                     4095, 4096, 4097, 12287, 12288, 12289, 13311, 13312, 13313, 20479, 20480, 20481, 32767, 32768, 32769, 40000])
    cuts = np.cumsum(lens).astype(np.uint64)
    d = corpus8[3:3 + int(cuts[-1])]
    zd = corpus.zdict()
    blob, offs = hmse_b200.compress(d, cuts, None, zd, ctx=ctx)
    _roundtrip(d, cuts, None, zd, blob, offs)
    blob, offs = hmse_b200.compress(d, cuts, None, b"", ctx=ctx)
    _roundtrip(d, cuts, None, b"", blob, offs)


def test_selection_order_and_repeats(ctx, corpus8):
    import hmse_b200
    d = corpus8[:1 << 20]
    cuts = oracle.chunk_c(d)
    sel = np.array([5, 0, 5, cuts.size - 1, 17, 3], dtype=np.uint64)
    zd = corpus.zdict()
    blob, offs = hmse_b200.compress(d, cuts, sel, zd, ctx=ctx)
    _roundtrip(d, cuts, sel.astype(np.int64), zd, blob, offs)
    empty, eo = hmse_b200.compress(d, cuts, np.zeros(0, np.uint64), zd, ctx=ctx)
    assert empty.size == 0 and eo.size == 1


def test_short_dictionary_and_level0(ctx, corpus8):
    import hmse_b200
    d = corpus8[:512 << 10]
    cuts = oracle.chunk_c(d)
    zd = corpus.zdict()[-1000:]
    blob, offs = hmse_b200.compress(d, cuts, None, zd, ctx=ctx)
    _roundtrip(d, cuts, None, zd, blob, offs)
    blob0, offs0 = hmse_b200.compress(d, cuts, None, zd, level=0, ctx=ctx)
    _roundtrip(d, cuts, None, zd, blob0, offs0)
    assert blob0.size > d.size


def test_deterministic_and_start0(ctx, corpus8):
    import hmse_b200
    d = corpus8[:2 << 20]
    cuts = oracle.chunk_c(d)
    zd = corpus.zdict()
    a, ao = hmse_b200.compress(d, cuts, None, zd, ctx=ctx)
    b, bo = hmse_b200.compress(d, cuts, None, zd, ctx=ctx)
    assert np.array_equal(a, b) and np.array_equal(ao, bo)
    c, co = hmse_b200.compress(d, cuts[4:], None, zd, start0=int(cuts[3]), ctx=ctx)
    outs = oracle.inflate_all(c, co, zd)
    assert b"".join(outs) == bytes(memoryview(d)[int(cuts[3]):])


def test_shifted_text_like_data(ctx, corpus8):
    # odd start offsets exercise the byte-unaligned staging of every chunk
    import hmse_b200
    zd = corpus.zdict()
    for off in (1, 2, 3):
        d = corpus8[off:off + (256 << 10)]
        cuts = oracle.chunk_c(d)
        blob, offs = hmse_b200.compress(d, cuts, None, zd, ctx=ctx)
        _roundtrip(d, cuts, None, zd, blob, offs)


def test_repetitive_data_is_not_pathologically_slow(ctx, corpus8):
    """A run of one byte puts every position of a 512-byte tile into ONE hash bucket: the bucket sort of parse_kernel
    must not fall back to a quadratic walk by a single thread there (it once did: 0.11 GB/s on zeros against 32 on text).
    Relative bound, generous: zeros and a 7-byte period compress at no less than 1/20 of the text rate."""
    import torch

    n = 8 << 20
    zd = ctx.stage(corpus.zdict())
    cuts = ctx.stage_u64(np.arange(8192, n + 1, 8192, dtype=np.uint64))

    def rate(data):
        d = ctx.stage(data)
        ctx.compress(d, cuts, None, zd)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        blob, offs = ctx.compress(d, cuts, None, zd)
        b.record()
        torch.cuda.synchronize()
        return n / a.elapsed_time(b), blob, offs

    text_rate, _, _ = rate(corpus8[:n])
    for name, data in (("zeros", np.zeros(n, dtype=np.uint8)),
                       ("period7", np.frombuffer((b"abcdefg" * (n // 7 + 1))[:n], dtype=np.uint8))):
        r, blob, offs = rate(data)
        assert r >= text_rate / 20, "%s: %.2f of the text rate" % (name, r / text_rate)
        hb, ho = blob.cpu().numpy(), offs.cpu().numpy().view(np.uint64)
        for k in (0, 1, cuts.numel() - 1):
            raw = zlib.decompressobj(zdict=corpus.zdict()).decompress(hb[int(ho[k]):int(ho[k + 1])].tobytes())
            assert raw == data[k * 8192:(k + 1) * 8192].tobytes()
