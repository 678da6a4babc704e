"""Inputs and expected streams for the byte-exact tests of the GPU DEFLATE encoder (tests/test_gpu_deflate_exact.py,
tests/test_deflate_model.py).  TEST INFRASTRUCTURE.

A case is one hmse_compress call: data, cut points, optional selection, preset dictionary, level, start0, and the
byte offset of the data pointer inside a 16-byte aligned buffer.  The expected stream of every selected chunk comes from
the CPU model (tests/model/deflate_model.cpp) with the kernel's parameters, or, for stored streams, from Python."""
import os
import zlib
from concurrent.futures import ThreadPoolExecutor

import ctypes as C
import numpy as np

from oracle import corpus

from .build import Params, build

# size classes of parse_kernel (csrc/deflate.cu NMAX_*) and their own-chunk candidate counts (OWN_*)
NMAX_SMALL, NMAX_MEDIUM, NMAX_LARGE = 13312, 20480, 32768
LONG_BLOCK, LONG_MAX_BLOCKS, STORED_MAX = 32768, 2048, 65535
DICT_CAP = 4


def size_class(n):
    return "small" if n <= NMAX_SMALL else "medium" if n <= NMAX_MEDIUM else "large" if n <= NMAX_LARGE else "long"


def own_of(n):
    return {"small": 2, "medium": 3, "large": 4, "long": 4}[size_class(n)]


def params(n, own=None, dict_cap=DICT_CAP, prev0=1):
    """The kernel's search for a chunk of n bytes (every block of a long chunk: the large class's 4 own candidates)."""
    return Params(hash_bytes=4, chain_own=own_of(n) if own is None else own, chain_dict=dict_cap, lazy=1, too_far=0,
                  dict_hash_bits=15, mode=2, min_len=0, hist=0, prev0=prev0)


def stored_stream(chunk, zd=b""):
    """zlib stream of stored blocks of at most 65535 bytes (an empty final block when the length is a multiple of
    65535), as the kernels write them for level 0, for long chunks that do not compress and beyond 2048 blocks."""
    chunk = bytes(chunk)
    n = len(chunk)
    nb = n // STORED_MAX + 1
    head = bytes([0x78, 0xBB]) + zlib.adler32(zd).to_bytes(4, "big") if zd else bytes([0x78, 0x9C])
    parts = [head]
    for b in range(nb):
        blk = chunk[b * STORED_MAX:(b + 1) * STORED_MAX]
        ln = len(blk)
        parts.append(bytes([1 if b == nb - 1 else 0, ln & 255, ln >> 8, ~ln & 255, (~ln >> 8) & 255]))
        parts.append(blk)
    parts.append(zlib.adler32(chunk).to_bytes(4, "big"))
    return b"".join(parts)


class Model:
    def __init__(self):
        self.lib = build()

    def stream(self, chunk, zd=b"", level=6, own=None, dict_cap=DICT_CAP, prev0=1):
        ch = np.ascontiguousarray(np.frombuffer(bytes(chunk), dtype=np.uint8))
        n = ch.size
        if level == 0:
            return stored_stream(ch, zd)
        zdn = np.frombuffer(zd, dtype=np.uint8) if zd else np.zeros(1, np.uint8)
        pr = params(n, own, dict_cap, prev0)
        out = np.zeros(n + 5 * (n // STORED_MAX + 1) + 64, dtype=np.uint8)
        if n <= NMAX_LARGE:
            r = self.lib.model_compress(ch.ctypes.data, n, zdn.ctypes.data, len(zd), C.byref(pr), out.ctypes.data, out.size,
                                        None)
        else:
            r = self.lib.model_compress_long(ch.ctypes.data, n, zdn.ctypes.data, len(zd), C.byref(pr), level,
                                             out.ctypes.data, out.size)
        assert r > 0, "model failed (%d) on a chunk of %d bytes" % (r, n)
        return out[:r].tobytes()

    def streams(self, chunks, zd=b"", level=6, **kw):
        """Streams of many chunks; ctypes drops the GIL, so they are computed by a thread per core."""
        with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
            return list(ex.map(lambda c: self.stream(c, zd, level, **kw), chunks))


class Case:
    def __init__(self, name, data, cuts, zd=b"", select=None, level=6, start0=0, ptr_off=0):
        self.name, self.zd, self.level, self.start0, self.ptr_off = name, bytes(zd), level, int(start0), ptr_off
        self.data = np.array(data, dtype=np.uint8)   # an own, writable copy (torch.from_numpy wants one)
        self.cuts = np.asarray(cuts, dtype=np.uint64)
        self.select = None if select is None else np.asarray(select, dtype=np.int64)

    def chunk(self, j):
        s = int(self.cuts[j - 1]) if j else self.start0
        return self.data[s:int(self.cuts[j])].tobytes()

    def order(self):
        """Chunk index of every output stream."""
        return np.arange(self.cuts.size) if self.select is None else self.select

    def expected(self, model, memo=None):
        """Expected streams in output order; the model runs once per distinct chunk (memo: shared across cases)."""
        memo = {} if memo is None else memo
        sel = self.order()
        distinct = sorted(set(sel.tolist()))
        keys = {j: (self.chunk(j), self.zd, self.level) for j in distinct}
        todo = [j for j in distinct if keys[j] not in memo]
        for j, s in zip(todo, model.streams([keys[j][0] for j in todo], self.zd, self.level)):
            memo[keys[j]] = s
        return [memo[keys[j]] for j in sel.tolist()]


# ---- inputs ------------------------------------------------------------------------------------------------------

def _rng(seed):
    return np.random.default_rng(seed)


def text(n, off=0):
    return corpus.generate(off + n)[off:]


def zdict():
    return corpus.zdict()


def binary_families(n, seed=1):
    """name -> n bytes: typed arrays as they sit in memory, random bytes, random bytes dense in 0xFE / 0xFF."""
    r = _rng(seed)
    m4, m2 = n // 4 + 1, n // 2 + 1
    fe = r.integers(0, 256, n, dtype=np.uint8)
    pick = r.random(n)
    fe[pick < 0.3] = 0xFE
    fe[(pick >= 0.3) & (pick < 0.6)] = 0xFF
    return {
        "int32": np.round(r.normal(0, 200, m4)).astype(np.int32).view(np.uint8)[:n],
        "int16": np.round(r.normal(0, 3000, m2)).astype(np.int16).view(np.uint8)[:n],
        "float32": np.cumsum(r.normal(0, 1, m4)).astype(np.float32).view(np.uint8)[:n],
        "random": r.integers(0, 256, n, dtype=np.uint8),
        "fe_ff": fe,
    }


def degenerate_families(n):
    """name -> n bytes that make long same-bucket groups (P3b's CTA-wide sort), long runs and the 258 cap."""
    out = {"zeros": np.zeros(n, np.uint8), "run_fe": np.full(n, 0xFE, np.uint8), "run_ff": np.full(n, 0xFF, np.uint8)}
    r = _rng(7)
    for p in (2, 3, 7, 64, 258, 259):
        out["period%d" % p] = np.resize(r.integers(0, 256, p, dtype=np.uint8), n)
    t = text(n).copy()
    pos = 0
    while pos < n:   # text broken by zero runs of 100 .. 3000 bytes
        pos += int(r.integers(200, 4000))
        t[pos:pos + int(r.integers(100, 3000))] = 0
        pos += 3000
    out["text_zero_runs"] = t
    return out


def sentinel_vectors():
    """The three hand-built vectors on which the run-head test at position 0 decides (prev0 of the model):
    (name, chunk, dictionary).  Each holds a 40-byte string S twice, where one copy is at position 0 of its side."""
    r = _rng(1)
    S = r.integers(0, 256, 40, dtype=np.uint8).tobytes()

    def fill(k):
        return r.integers(0, 256, k, dtype=np.uint8).tobytes()

    return [
        # own source at chunk position 0 (kernel: preceded by 0xFE) against a position preceded by 0xFE
        ("own_q0_after_fe", S + fill(500) + b"\xfe" + S + fill(100), b""),
        # chunk position 0 (0xFE before it) against a dictionary position preceded by 0xFE
        ("chunk_p0_dict_after_fe", S + fill(500), fill(300) + b"\xfe" + S + fill(300)),
        # dictionary position 0 (0xFF before it) against a chunk position preceded by 0xFF
        ("dict_j0_chunk_after_ff", fill(500) + b"\xff" + S + fill(100), S + fill(600)),
    ]


def sentinel_long_vectors():
    """The first two situations between block 1 of a long chunk and block 0, its dictionary (or inside block 1).  The
    third cannot arise there: only block position 0 reaches position 0 of the previous block (distance 32768), and the
    sentinels before the two differ.  The filler is text, so that the chunk is coded rather than stored."""
    r = _rng(2)
    S = r.integers(0, 256, 40, dtype=np.uint8).tobytes()
    src = text(4 * LONG_BLOCK, 2 << 20).tobytes()
    used = [0]

    def fill(k):
        used[0] += k
        return src[used[0] - k:used[0]]

    B = LONG_BLOCK
    return [
        ("long_own_q0_after_fe", fill(B) + S + fill(500) + b"\xfe" + S + fill(100)),
        ("long_block_p0_prev_after_fe", fill(300) + b"\xfe" + S + fill(B - 341) + S + fill(500)),
    ]


def _cuts(lens, start0=0):
    return (start0 + np.cumsum(np.asarray(lens, dtype=np.int64))).astype(np.uint64)


def _cat(parts):
    parts = [np.frombuffer(p, np.uint8) if isinstance(p, bytes) else np.asarray(p, np.uint8) for p in parts]
    return np.concatenate(parts), _cuts([p.size for p in parts])


def family_dicts():
    import oracle
    zd = zdict()
    big = text(3 << 20)
    t = big[:256 << 10]
    cuts = oracle.chunk_c(t)
    long_zd = (zd + text(8192, 1 << 20).tobytes())[-32767:]
    # 3 MiB of CDC chunks of corpus text with and without the text dictionary: the product's own workload
    cases = [Case("dict_text", big, oracle.chunk_c(big), zd), Case("dict_none", big[:1 << 20], oracle.chunk_c(big[:1 << 20]), b"")]
    for k in (1, 3, 4, 5, 1000):
        cases.append(Case("dict_%d" % k, t, cuts, zd[-k:]))
    cases.append(Case("dict_32767", t, cuts, long_zd))
    # the data itself as the dictionary: the first chunks repeat it, so matches end where the dictionary ends
    cases.append(Case("dict_self", t, cuts, t[:32768].tobytes()))
    return cases


LENGTHS = list(range(9)) + [13311, 13312, 13313, 20479, 20480, 20481, 32767, 32768]


def family_lengths():
    zd = zdict()
    t = text(len(LENGTHS) * 32768, 12345)
    cases = []
    for o in range(16):   # first chunk at start offsets 0..15 (all staging alignments), the rest follow on
        cases.append(Case("lengths_start%d" % o, t[:o + sum(LENGTHS)], _cuts(LENGTHS, o), zd, start0=o))
    for po in (4, 8, 12):   # a data pointer that is only 4-byte aligned: the first chunk is staged word by word
        for o in (0, 3):
            cases.append(Case("lengths_ptr%d_start%d" % (po, o), t[:o + sum(LENGTHS)], _cuts(LENGTHS, o), b"", start0=o,
                              ptr_off=po))
    return cases


def _mixed_cuts(n, seed):
    """CDC-like ragged cut points that cover all three size classes."""
    r = _rng(seed)
    lens, tot = [], 0
    while tot < n:
        k = int(r.choice([r.integers(1, 4000), r.integers(4000, NMAX_SMALL + 1), r.integers(NMAX_SMALL + 1, NMAX_MEDIUM + 1),
                          r.integers(NMAX_MEDIUM + 1, NMAX_LARGE + 1)]))
        k = min(k, n - tot)
        lens.append(k)
        tot += k
    return _cuts(lens)


def family_binary():
    import oracle
    zd = zdict()
    cases = []
    for i, (name, d) in enumerate(binary_families(512 << 10).items()):
        cases.append(Case("bin_%s_cdc" % name, d, oracle.chunk_c(d), zd if i % 2 else b""))
        cases.append(Case("bin_%s_mixed" % name, d, _mixed_cuts(d.size, i), b"" if i % 2 else zd))
    for name, ch, dct in sentinel_vectors():
        cases.append(Case("sentinel_" + name, np.frombuffer(ch, np.uint8), _cuts([len(ch)]), dct))
    return cases


def family_degenerate():
    zd = zdict()
    lens = [1000, 5000, 8192, 13312, 13313, 16000, 20480, 20481, 25000, 32767, 32768]
    cases = []
    for i, (name, d) in enumerate(degenerate_families(sum(lens)).items()):
        cases.append(Case("degen_%s" % name, d, _cuts(lens), b""))
        cases.append(Case("degen_%s_dict" % name, np.roll(d, 333), _cuts(lens), zd))
    return cases


LONG_LENS = [32769, 65535, 65536, 65537, 3 * 32768 + 5, 1 << 20]


def family_long():
    zd = zdict()
    n = sum(LONG_LENS)
    bins = binary_families(n, seed=5)
    r = _rng(11)
    # text, binary and random chunks of every long length in one call: 135 blocks, more than one batch of 96
    d = np.concatenate([text(n, 77), bins["int16"], bins["random"]])
    cuts = _cuts(LONG_LENS * 3)
    cases = [Case("long_mixed_dict", d, cuts, zd), Case("long_mixed_nodict", d, cuts, b"")]
    z = np.concatenate([np.zeros(100000, np.uint8), np.resize(r.integers(0, 256, 259, dtype=np.uint8), 70000)])
    cases.append(Case("long_degenerate", z, _cuts([100000, 70000]), b""))
    sd, sc = _cat([v for _, v in sentinel_long_vectors()])
    cases.append(Case("long_sentinel_vectors", sd, sc, b""))
    cases.append(Case("long_sentinel_vectors_dict", sd, sc, zd))
    # level 0: stored blocks for every class (expected streams built in Python)
    lv = np.concatenate([text(300000, 5), bins["int32"][:300000]])
    lc = _cuts([0, 1, 100, 13313, 32768, 32769, 65535, 65536, 65537, 70000] + [5000] * 10)
    lc = lc[lc <= lv.size]
    cases.append(Case("level0_dict", lv, lc, zd, level=0))
    cases.append(Case("level0_nodict", lv, lc, b"", level=0))
    return cases


def family_batches():
    """A selection that repeats a few chunks: 32769 small, 16385 medium and 8193 large entries (one more than a batch
    of each class), shuffled, reversed, and with start0 > 0."""
    zd = zdict()
    bins = binary_families(32768, seed=9)
    parts = [text(8000, 3), bins["int32"][:6000], np.zeros(13312, np.uint8),        # small
             text(16000, 99), bins["int16"][:20480],                               # medium
             text(30000, 555), bins["random"][:32768]]                             # large
    pad = 7
    data = np.concatenate([np.full(pad, 0x55, np.uint8)] + parts)
    cuts = _cuts([p.size for p in parts], pad)
    r = _rng(13)
    sel = np.concatenate([r.integers(0, 3, 32769), r.integers(3, 5, 16385), r.integers(5, 7, 8193)])
    sel = sel[r.permutation(sel.size)]
    return [Case("batch_shuffled", data, cuts, zd, select=sel, start0=pad),
            Case("batch_reversed", data, cuts, b"", select=np.sort(sel)[::-1].copy(), start0=pad)]


def dict_cache_dicts():
    """Dictionaries A and B, and A2: A with +1, -2, +1 on three adjacent bytes - same length and Adler-32 as A."""
    a = zdict()
    b = text(len(a), 3 << 20).tobytes()
    i = len(a) // 2
    while not (a[i] < 255 and a[i + 1] >= 2 and a[i + 2] < 255):
        i += 1
    a2 = bytearray(a)
    a2[i] += 1
    a2[i + 1] -= 2
    a2[i + 2] += 1
    a2 = bytes(a2)
    assert len(a2) == len(a) and zlib.adler32(a2) == zlib.adler32(a) and a2 != a
    return a, b, a2, i


def family_dict_cache():
    a, b, a2, i = dict_cache_dicts()
    # chunks that quote the dictionaries around the three changed bytes, then text
    quote = np.frombuffer(a[i - 2000:i + 2000] + a2[i - 1000:i + 1000] + b[:3000], np.uint8)
    t = text(60000, 4321)
    d = np.concatenate([quote, t])
    cuts = _cuts([4000, 2000, 3000, 20000, 40000])
    return [Case("cache_A", d, cuts, a), Case("cache_B", d, cuts, b), Case("cache_A_again", d, cuts, a),
            Case("cache_A2_same_adler", d, cuts, a2), Case("cache_A_last", d, cuts, a)]


FAMILIES = {
    "dicts": family_dicts,
    "lengths": family_lengths,
    "binary": family_binary,
    "degenerate": family_degenerate,
    "long": family_long,
    "batches": family_batches,
    "dict_cache": family_dict_cache,
}
