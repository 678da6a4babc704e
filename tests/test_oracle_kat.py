"""CPU tests pinning the oracle (oracle/): public known-answer vectors for the third-party
primitives the spec names but does not vendor (SHA-256 - mbedtls README.md:2543; MurmurHash3 -
murmur3.h README.md:2573; zlib/miniz README.md:2352), hand-checked FastCDC conventions, the
committed golden fixtures, and the properties the spec's validation plan demands
(VALIDATION_METHODS.md:115-128, 257; README.md:1254, 2234)."""
import hashlib
import json
import os
import zlib

import numpy as np
import pytest

import oracle
from oracle import corpus
from oracle.config import CDCConfig, M64

HERE = os.path.dirname(os.path.abspath(__file__))


# ---- public known-answer vectors (SURVEY.md §4) -------------------------------------------------
def test_sha256_kat():
    d = oracle.digest(b"abc", np.array([3], dtype=np.uint64))
    assert d[0].tobytes().hex() == "ba7816bf8f01cfea414140de5dae2223b00361a396177a9cb410ff61f20015ad"
    d = oracle.digest(b"", np.array([0], dtype=np.uint64))
    assert d[0].tobytes().hex() == "e3b0c44298fc1c149afbf4c8996fb92427ae41e4649b934ca495991b7852b855"


@pytest.mark.parametrize("key,seed,want", [
    (b"", 0, 0x00000000), (b"", 1, 0x514E28B7), (b"", 0xFFFFFFFF, 0x81F16F39), (b"\xff\xff\xff\xff", 0, 0x76293B50),
    (b"\x21\x43\x65\x87", 0, 0xF55B516B), (b"\x21\x43\x65\x87", 0x5082EDEE, 0x2362F9DE), (b"abc", 0, 0xB3DD93FA),
    (b"Hello, world!", 0x9747B28C, 0x24884CBA), (b"Albe", 0, 0xD1825B61), (b"Albe", 1, 0xB9F244D2),
    (b"Albe", 127, 0x0DA11A3B), (b"Albe", 128, 0xB1704FF1)])
def test_murmur3_kat(key, seed, want):
    assert oracle.murmur3_32(key, seed) == want


def test_murmur3_c_port_equals_python():
    lib = oracle.cdc.ref_lib()
    lib.hmse_ref_murmur3_4.restype = __import__("ctypes").c_uint32
    for k, s in [(0x65626C41, 0), (0x65626C41, 1), (0, 0), (0xFFFFFFFF, 0x5082EDEE), (0x87654321, 7)]:
        key = int(k).to_bytes(4, "little")
        assert lib.hmse_ref_murmur3_4(k, s) == oracle.murmur3_32(key, s)


def test_minhash_matches_murmur_definition():
    data = np.frombuffer(b"Albert Einstein was a theoretical physicist.", dtype=np.uint8)
    cuts = np.array([data.size], dtype=np.uint64)
    sig = oracle.minhash(data, cuts)
    raw = data.tobytes()
    for p in (0, 1, 63, 127):
        seed = p + 1
        want = min(oracle.murmur3_32(raw[i:i + 4], seed) for i in range(len(raw) - 3))
        assert int(sig[0, p]) == want
    assert np.array_equal(sig, oracle.minhash_c(data, cuts))
    short = oracle.minhash(data[:3], np.array([3], dtype=np.uint64))
    assert (short == 0xFFFFFFFF).all()      # SURVEY.md §0.2 C10


def test_murmur3_and_minhash_against_an_independent_implementation():
    """MurmurHash3_x86_32 is a third-party primitive the spec names (murmur3.h, README.md:2573, 2591) and does not
    vendor.  scikit-learn ships its own C++ copy of Appleby's function (sklearn.utils.murmurhash3_32, written by other
    people): the oracle's hash (random keys of every length 0..40, random seeds) and whole MinHash signatures - NumPy
    and C restatements - must equal what that implementation gives, so the pin does not rest on twelve vectors alone.
    Its answers are stored in tests/golden/murmur3_sklearn.json (tests/golden/make_murmur3_golden.py), so the pin holds
    without scikit-learn; where it is installed, the stored answers are recomputed with it and must be the same."""
    with open(os.path.join(HERE, "golden", "murmur3_sklearn.json")) as f:
        golden = json.load(f)
    assert len(golden["hashes"]) == 41 * 8
    for key, seed, want in golden["hashes"]:
        assert oracle.murmur3_32(bytes.fromhex(key), seed) == want
    mh = golden["minhash"]
    data = corpus.generate(mh["cuts"][-1])
    assert hashlib.sha256(data.tobytes()).hexdigest() == mh["input_sha256"], "corpus generator drifted"
    cuts = np.array(mh["cuts"], dtype=np.uint64)      # a 3-byte chunk among them
    sig = oracle.minhash(data, cuts)
    assert np.array_equal(sig, oracle.minhash_c(data, cuts))
    assert len(mh["mins"]) == cuts.size * 3
    for j, p, want in mh["mins"]:
        assert int(sig[j, p]) == want
    try:
        import sklearn.utils  # noqa: F401
    except ImportError:
        return
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_murmur3_golden", os.path.join(HERE, "golden", "make_murmur3_golden.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    assert gen.vectors() == golden


def test_zlib_preset_dictionary_framing():
    zd = corpus.zdict()
    data = corpus.generate(20000)
    blob, offs = oracle.compress(data, np.array([20000], dtype=np.uint64), [0], zd)
    assert blob[0] == 0x78 and blob[1] == 0xBB
    assert int.from_bytes(blob[2:6].tobytes(), "big") == zlib.adler32(zd)
    assert int.from_bytes(blob[-4:].tobytes(), "big") == zlib.adler32(data.tobytes())
    assert oracle.inflate_all(blob, offs, zd)[0] == data.tobytes()
    with pytest.raises(Exception):
        oracle.inflate_all(blob, offs, b"")        # needs the dictionary


# ---- FastCDC conventions ----------------------------------------------------------------------------
def test_gear_table_pinned():
    g = oracle.gear_table()
    assert g.dtype == np.uint64 and g.size == 256 and len(set(g.tolist())) == 256
    golden = json.load(open(os.path.join(HERE, "golden", "hotpath_golden.json")))
    assert hashlib.sha256(g.tobytes()).hexdigest() == golden["gear_sha256"]
    assert bin(oracle.PAPER_MASK_S).count("1") == 15 and bin(oracle.PAPER_MASK_L).count("1") == 11


def test_cut_convention_hand_computed():
    """The byte that completes the match starts the NEXT chunk (oracle/cdc.py header).  A Gear
    table with one entry 0 makes a zero run hash to 0 (clears every mask), so the hit is forced at
    the first tested position."""
    cfg = CDCConfig(64, 128, 512, 0x0000F00000000000, 0x0000300000000000)
    gear = cfg.gear.tolist()
    zb = 7
    data = np.full(2000, zb, dtype=np.uint8)
    g2 = list(gear)
    # emulate: use next_cut with a patched table where Gear[zb] == 0
    g2[zb] = 0
    assert oracle.next_cut(data.tolist(), 0, data.size, cfg, g2) == cfg.min_size      # fp=0 at i=min -> return i=min
    assert oracle.next_cut(data.tolist(), 100, data.size, cfg, g2) == 100 + cfg.min_size
    # no candidate at all -> forced cut at max_size: with every Gear entry == 1<<47 the newest byte
    # always sets bit 47 (older bytes only reach higher bits), so a mask containing bit 47 never clears
    cfg47 = CDCConfig(64, 128, 512, 1 << 47, 1 << 47)
    g3 = [1 << 47] * 256
    assert oracle.next_cut(data.tolist(), 0, data.size, cfg47, g3) == cfg47.max_size
    assert oracle.next_cut(data.tolist(), 300, data.size, cfg47, g3) == 300 + cfg47.max_size
    # tail no longer than min_size -> the cut is the end of the stream
    assert oracle.next_cut(data.tolist(), 1990, data.size, cfg, gear) == data.size
    assert oracle.next_cut(data.tolist(), data.size - cfg.min_size, data.size, cfg, gear) == data.size


def test_three_chunkers_agree():
    for seed, n in [(1, 0), (2, 1), (3, 2047), (4, 2048), (5, 2049), (6, 70000), (7, 200000)]:
        d = corpus.random_bytes(n, seed) if n else np.zeros(0, np.uint8)
        a, b, c = oracle.chunk_naive(d), oracle.chunk(d), oracle.chunk_c(d)
        assert np.array_equal(a, b) and np.array_equal(a, c)
        if n:
            assert int(a[-1]) == n and (np.diff(a.astype(np.int64)) > 0).all()
    t = corpus.generate(300000)
    for cfg in (CDCConfig(), CDCConfig.for_avg(4096), CDCConfig.for_avg(16384, 1)):
        assert np.array_equal(oracle.chunk_naive(t, cfg), oracle.chunk(t, cfg))
        assert np.array_equal(oracle.chunk(t, cfg), oracle.chunk_c(t, cfg))


def test_three_chunkers_agree_on_random_geometries():
    """Property test (hypothesis): the literal byte loop of Algorithm 1 (chunk_naive, the ground truth of the oracle), the
    NumPy restatement and the C restatement give the same cut list for random min / avg / max, random masks (any bits
    of the 64, also low ones and masks with common bits), another Gear seed, and contents from random bytes to runs of
    one byte and short periods - the inputs where `normal point`, `max` and end-of-stream rules meet."""
    hyp = pytest.importorskip("hypothesis")
    st = pytest.importorskip("hypothesis.strategies")

    @st.composite
    def cases(draw):
        mn = draw(st.integers(64, 600))
        av = draw(st.integers(mn, 1500))
        mx = draw(st.integers(av, 4000))
        ms = draw(st.integers(1, M64)) & draw(st.integers(1, M64)) or 1 << 40
        ml = draw(st.integers(1, M64)) & draw(st.integers(1, M64)) & draw(st.integers(1, M64)) or 1 << 33
        cfg = CDCConfig(mn, av, mx, ms, ml, draw(st.sampled_from([0x484D5345, 1, 0xDEADBEEF])))
        n = draw(st.integers(0, 12000))
        kind = draw(st.sampled_from(["random", "zeros", "period", "two", "text"]))
        seed = draw(st.integers(0, 2 ** 31))
        rng = np.random.default_rng(seed)
        if kind == "random":
            d = rng.integers(0, 256, n, dtype=np.uint8)
        elif kind == "zeros":
            d = np.full(n, draw(st.integers(0, 255)), dtype=np.uint8)
        elif kind == "period":
            d = np.resize(rng.integers(0, 256, draw(st.integers(1, 97)), dtype=np.uint8), n)
        elif kind == "two":
            d = rng.integers(0, 2, n, dtype=np.uint8) * 255
        else:
            d = corpus.generate(n + 1)[:n]
        return cfg, np.ascontiguousarray(d, dtype=np.uint8)

    @hyp.settings(max_examples=200, deadline=None, derandomize=True,
                  suppress_health_check=list(hyp.HealthCheck))
    @hyp.given(cases())
    def check(case):
        cfg, d = case
        a, b, c = oracle.chunk_naive(d, cfg), oracle.chunk(d, cfg), oracle.chunk_c(d, cfg)
        assert np.array_equal(a, b) and np.array_equal(a, c)
        if d.size:
            lens = np.diff(np.concatenate([[0], a]).astype(np.int64))
            assert int(a[-1]) == d.size and (lens > 0).all() and lens.max() <= cfg.max_size
            assert lens.size == 1 or lens[:-1].min() >= cfg.min_size

    check()


def test_chunk_size_distribution_and_bounds():
    # README.md:1137, 2510-2514 acceptance: min/max respected; mean near the target
    d = corpus.generate(8 << 20)
    for cfg, lo, hi in ((CDCConfig(), 0.85, 1.35), (CDCConfig.for_avg(4096), 0.85, 1.35)):
        cuts = oracle.chunk_c(d, cfg)
        lens = np.diff(np.concatenate([[0], cuts]).astype(np.int64))
        assert lens[:-1].min() >= cfg.min_size and lens.max() <= cfg.max_size
        assert lo * cfg.avg_size <= lens.mean() <= hi * cfg.avg_size


def test_shift_resistance():
    d = corpus.generate(4 << 20)
    a = oracle.chunk_c(d).astype(np.int64)
    b = oracle.chunk_c(np.concatenate([corpus.random_bytes(100, 7), d])).astype(np.int64) - 100
    assert np.intersect1d(a, b).size >= 0.99 * a.size       # README.md:1254


def test_shard_walk_equals_stream():
    d = corpus.generate(1 << 20)
    cfg = CDCConfig()
    want = oracle.chunk(d, cfg)
    half = 500000
    c0, ex = oracle.cdc.chunk_shard(d[:half + cfg.max_size], cfg, 0, half, False)
    c1, _ = oracle.cdc.chunk_shard(d[half:], cfg, ex - half, d.size - half, True)
    assert np.array_equal(np.concatenate([c0, c1 + np.uint64(half)]), want)


# ---- golden fixtures --------------------------------------------------------------------------------
def test_oracle_matches_committed_golden():
    import sys
    sys.path.insert(0, os.path.join(HERE, "golden"))
    import make_golden
    golden = json.load(open(os.path.join(HERE, "golden", "hotpath_golden.json")))
    ins = make_golden.inputs()
    src = {"text": ins["text"], "text_4k": ins["text"], "dup": ins["dup"], "random": ins["random"]}
    assert hashlib.sha256(corpus.zdict()).hexdigest() == golden["zdict_sha256"]
    for c in golden["cases"]:
        data = src[c["name"]]
        assert hashlib.sha256(data.tobytes()).hexdigest() == c["input_sha256"], "corpus generator drifted"
        cfg = CDCConfig(*c["cfg"])
        cuts = oracle.chunk_c(data, cfg)
        assert cuts.tolist() == c["cuts"]
        dg = oracle.digest(data, cuts)
        assert hashlib.sha256(dg.tobytes()).hexdigest() == c["digests_sha256"]
        assert oracle.dedup(dg)[0].tolist() == c["canon"]
        sig = oracle.minhash_c(data, cuts[:3])
        assert sig[0].tolist() == c["sig0"]
        assert oracle.band_keys(sig)[0].tolist() == c["keys0"]


# ---- spec properties -----------------------------------------------------------------------------------
def test_dedup_five_copies():
    one = corpus.generate(1 << 20)
    d = np.tile(one, 5)
    cuts = oracle.chunk_c(d)
    canon, first = oracle.dedup(oracle.digest(d, cuts))
    lens = np.diff(np.concatenate([[0], cuts]).astype(np.int64))
    assert lens[first].sum() <= 1.1 * one.size          # README.md:1210, 1299-1315
    assert (canon <= np.arange(canon.size)).all() and (canon[first] == np.flatnonzero(first)).all()


def test_minhash_estimates_jaccard():
    rng = np.random.default_rng(5)
    base = corpus.generate(20000)
    for frac in (0.02, 0.2):
        other = base.copy()
        idx = rng.choice(base.size, int(frac * base.size / 8), replace=False)
        other[idx] = rng.integers(97, 123, idx.size)
        both = np.concatenate([base, other])
        sig = oracle.minhash_c(both, np.array([base.size, both.size], dtype=np.uint64))

        def shingles(x):
            b = x.astype(np.uint32)
            return set((b[:-3] | (b[1:-2] << 8) | (b[2:-1] << 16) | (b[3:] << 24)).tolist())
        sa, sb = shingles(base), shingles(other)
        jac = len(sa & sb) / len(sa | sb)
        agree = float((sig[0] == sig[1]).mean())
        sigma = (jac * (1 - jac) / 128) ** 0.5
        assert abs(agree - jac) <= 4 * sigma + 0.02      # README.md:1359-1373


def test_lsh_collision_probability_formula():
    # README.md:2234: P = 1 - (1 - s^r)^b; checked by Monte-Carlo on synthetic signatures
    rng = np.random.default_rng(11)
    cfg = oracle.SimConfig()
    for s in (0.5, 0.8):
        n = 4000
        a = rng.integers(0, 1 << 32, (n, 128), dtype=np.uint64).astype(np.uint32)
        b = a.copy()
        flip = rng.random((n, 128)) >= s
        b[flip] = rng.integers(0, 1 << 32, int(flip.sum()), dtype=np.uint64).astype(np.uint32)
        hit = (oracle.band_keys(a, cfg) == oracle.band_keys(b, cfg)).any(axis=1).mean()
        want = 1 - (1 - s ** cfg.rows) ** cfg.bands
        assert abs(hit - want) < 0.03


def test_buckets_sorted_and_complete():
    keys = np.array([[3, 1], [3, 0], [2, 1]], dtype=np.uint64)
    band, key, ids = oracle.buckets(keys, id_base=10)
    assert band.tolist() == [0, 0, 0, 1, 1, 1]
    assert key.tolist() == [2, 3, 3, 0, 1, 1] and ids.tolist() == [12, 10, 11, 11, 10, 12]


def test_corpus_redundancy_mix():
    d = corpus.generate(16 << 20)
    cuts = oracle.chunk_c(d)
    _, first = oracle.dedup(oracle.digest(d, cuts))
    assert 0.55 <= first.mean() <= 0.95           # duplicates exist, most content is unique at this size
    hi = corpus.generate(16 << 20, corpus.CorpusConfig.high_redundancy())
    cuts = oracle.chunk_c(hi)
    _, first_hi = oracle.dedup(oracle.digest(hi, cuts))
    assert first_hi.mean() < first.mean()


def test_compression_ratio_with_dictionary_beats_without():
    d = corpus.generate(1 << 20)
    cuts = oracle.chunk_c(d)
    sel = np.arange(cuts.size)
    with_d, _ = oracle.compress(d, cuts, sel, corpus.zdict())
    without, _ = oracle.compress(d, cuts, sel, b"")
    assert with_d.size < 0.8 * without.size and d.size / with_d.size >= 2.5      # README.md:2417-2420 ratio >= 2.5


def test_archive_records_and_pure_zlib_restore():
    # oracle/archive.py against hand-checked field values and a zlib-only round trip
    import zlib
    from oracle import archive
    zd = corpus.zdict()
    data = corpus.generate(600000)
    data = np.concatenate([data, data[:200000]])
    cuts = oracle.chunk(data)
    dg = oracle.digest(data, cuts)
    canon, first = oracle.dedup(dg)
    sel = np.flatnonzero(first)
    blob, offs = oracle.compress(data, cuts, sel, zd)
    idx, ptr = archive.records(dg, canon, cuts, sel, offs)
    assert idx.shape == (sel.size, 40) and ptr.shape == (cuts.size, 8)
    k = 3
    assert idx[k, :32].tobytes() == dg[sel[k]].tobytes()
    assert int.from_bytes(idx[k, 32:36].tobytes(), "little") == int(offs[k]) >> 9
    assert int.from_bytes(idx[k, 36:38].tobytes(), "little") == int(offs[k + 1] - offs[k])
    assert int.from_bytes(idx[k, 38:40].tobytes(), "little") == int((canon == sel[k]).sum())
    i = int(np.flatnonzero(~first)[0])                       # a duplicate points at its first occurrence
    s = int(np.searchsorted(sel, canon[i]))
    assert int.from_bytes(ptr[i, 0:4].tobytes(), "little") * 512 + int.from_bytes(ptr[i, 4:6].tobytes(), "little") == int(offs[s])
    assert int.from_bytes(ptr[i, 6:8].tobytes(), "little") + 1 == int(cuts[i] - cuts[i - 1])
    buf = archive.pack(zd, idx, ptr, blob, data.size)
    assert buf[:8] == b"HMSEARC1" and archive.restore(buf) == data.tobytes()


def test_digest_mt_and_dedup_fast_equal_the_plain_oracle():
    """The threaded / sort-based forms used for the full-size parity checks are the same functions."""
    from oracle import corpus
    d = corpus.generate(3 << 20)
    d = np.concatenate([d, d[:1 << 20], d[(1 << 19):(3 << 19)]])
    cuts = oracle.chunk_c(d)
    a = oracle.digest(d, cuts)
    assert np.array_equal(a, oracle.digest_mt(d, cuts)) and np.array_equal(a, oracle.digest_mt(d, cuts, threads=3))
    assert np.array_equal(oracle.digest(d, cuts[5:], start0=int(cuts[4])), oracle.digest_mt(d, cuts[5:], start0=int(cuts[4])))
    c1, f1 = oracle.dedup(a)
    c2, f2 = oracle.dedup_fast(a)
    assert np.array_equal(c1, c2) and np.array_equal(f1, f2) and 0 < f1.sum() < f1.size
    e = oracle.dedup_fast(np.zeros((0, 32), dtype=np.uint8))
    assert e[0].size == 0 and e[1].size == 0
