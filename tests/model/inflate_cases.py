"""Streams for the exact decoder tests: every RFC 1950 / 1951 feature the read path must decode as stock zlib does,
valid and malformed, written with `deflate_writer` (TEST INFRASTRUCTURE).

A family is a list of groups; a group is one preset dictionary and its cases, which the GPU test decodes in one
`hmse_inflate` call.  A case carries its stream, the output length the caller expects, and a label: True (zlib
inflates it to `want`, the bytes its tokens stand for), False (zlib rejects it) or None (the damaged-stream family,
where zlib alone decides).  `zlib_verdict` is the reference: stock zlib plus the stricter contract of the read path."""
import zlib

import numpy as np

from tests.model import deflate_writer as W
from tests.model.inflate_tokens import _DIST_BASE, _DIST_EXTRA, _LEN_BASE, _LEN_EXTRA, read_zlib


def zlib_verdict(stream, zdict, expected_len):
    """The bytes `stream` inflates to under stock zlib, or None when the read path must reject it: FDICT set iff a
    dictionary is passed (zlib itself would ignore a dictionary the stream does not ask for), exactly one stream with
    nothing after its trailer, and exactly `expected_len` bytes of output."""
    stream = bytes(stream)
    if len(stream) < 2 or bool(stream[1] & 0x20) != bool(zdict):
        return None
    d = zlib.decompressobj(zdict=zdict) if zdict else zlib.decompressobj()
    try:
        out = d.decompress(stream)
    except zlib.error:
        return None
    if not d.eof or d.unused_data or len(out) != expected_len:
        return None
    return out


def describe(stream):
    """One line on the structure of a stream, or on why the token reader cannot read it."""
    try:
        s = read_zlib(stream)
    except (ValueError, IndexError) as e:
        return "read_zlib: %s" % e
    parts = []
    for b in s["blocks"][:4]:
        if b["type"] == 2:
            parts.append("dynamic HLIT %d HDIST %d HCLEN %d, max lengths %d / %d, %d tokens" % (
                b["hlit"], b["hdist"], b["hclen"], max(b["lit_lens"]), max(b["dist_lens"]), len(b["tokens"])))
        else:
            parts.append("%s, %d tokens" % ({0: "stored", 1: "fixed"}[b["type"]], len(b["tokens"])))
    more = " ..." if len(s["blocks"]) > 4 else ""
    return "%d bytes, %d block(s): %s%s" % (len(stream), len(s["blocks"]), "; ".join(parts), more)


class Case:
    def __init__(self, name, stream, out_len, valid, want=None, status=None):
        self.name, self.stream, self.out_len, self.valid = name, bytes(stream), int(out_len), valid
        self.want = want           # what zlib must inflate a valid case to
        self.status = status       # the status code the kernel's documentation fixes for this case, if any


class Group:
    def __init__(self, name, zd, cases):
        self.name, self.zd, self.cases = name, bytes(zd), cases


def _valid(name, blocks, zd=b"", **kw):
    s, raw = W.zlib_stream(blocks, zd, **kw)
    return Case(name, s, len(raw), True, raw)


def _invalid(name, blocks, zd=b"", out_len=None, **kw):
    s, raw = W.zlib_stream(blocks, zd, **kw)
    return Case(name, s, len(raw or b"") if out_len is None else out_len, False)


def _rng(seed):
    return np.random.default_rng(seed)


def _bytes(rng, n):
    return rng.integers(0, 256, n, dtype=np.uint8).tobytes()


def dict32k():
    return _bytes(_rng(32768), 32768)


def _match(rng, lsym, dsym):
    """A (length, distance) pair coded with length symbol lsym and distance symbol dsym, random extra bits (284
    stays below 258, which would be coded with 285)."""
    le, de = _LEN_EXTRA[lsym - 257], _DIST_EXTRA[dsym]
    lx = int(rng.integers(0, (1 << le) - (lsym == 284)))
    return (_LEN_BASE[lsym - 257] + lx, _DIST_BASE[dsym] + int(rng.integers(0, 1 << de)))


def tokens_using(lit_lens, dist_lens, rng):
    """Tokens that use every symbol the two codes hold, in random order; distances need a 32 KiB window."""
    lits = [s for s in range(min(256, len(lit_lens))) if lit_lens[s]]
    lsyms = [s for s in range(257, min(286, len(lit_lens))) if lit_lens[s]]
    dsyms = [d for d in range(min(30, len(dist_lens))) if dist_lens[d]]
    toks = list(lits)
    if lsyms and dsyms:
        for i in range(max(len(lsyms), len(dsyms))):
            toks.append(_match(rng, lsyms[i % len(lsyms)], dsyms[i % len(dsyms)]))
    order = rng.permutation(len(toks))
    return [toks[i] for i in order]


def _perm(lens, rng):
    return [lens[i] for i in rng.permutation(len(lens))]


def _lit_code(syms, n=286):
    """A complete literal/length code over `syms` (end-of-block is added), balanced."""
    syms = sorted(set(syms) | {256})
    lens = [0] * n
    for s, ln in zip(syms, W.balanced_lens(len(syms))):
        lens[s] = ln
    return lens


def _dyn(name, lit, dist, zd, rng, valid=True, tokens=None, **kw):
    toks = tokens_using(lit, dist, rng) if tokens is None else tokens
    blk = W.dynamic(toks, lit, dist, final=1, **kw)
    return (_valid if valid else _invalid)(name, [blk], zd)


# ---- families --------------------------------------------------------------------------------------------------

def family_code_shapes():
    zd, rng, cases = dict32k(), _rng(1), []
    for lm, dm, perm in [(10, 8, 1), (11, 9, 1), (15, 15, 1), (10, 15, 1), (15, 8, 1), (11, 8, 1), (15, 15, 0),
                         (10, 8, 0), (11, 9, 0)]:
        lit, dist = W.spine_lens(286, lm), W.spine_lens(30, dm)
        if perm:
            lit, dist = _perm(lit, rng), _perm(dist, rng)
        cases.append(_dyn("lit max %d, dist max %d, %s" % (lm, dm, "shuffled" if perm else "in order"), lit, dist, zd, rng))
    base = _lit_code(list(range(97, 123)) + [257, 262, 270, 284, 285])
    for k in (0, 4, 29):
        dist = [0] * (k + 1)
        dist[k] = 1
        cases.append(_dyn("single distance code %d of length 1" % k, base, dist, zd, rng))
    lit = _lit_code(range(32, 127))
    cases.append(_dyn("all-literal block, HDIST 1 with no distance code", lit, [0], zd, rng))
    cases.append(_dyn("all-literal block, 30 distance lengths all 0", lit, [0] * 30, zd, rng))
    eob = [0] * 257
    eob[256] = 1
    cases.append(_dyn("end-of-block alone at length 1, final", eob, [0], zd, rng, tokens=[]))
    cases.append(_valid("end-of-block alone at length 1, then a fixed block",
                        [W.dynamic([], eob, [0]), W.fixed(b"after", final=1)], zd))
    cases.append(_valid("end-of-block alone at length 1, one distance code of length 1",
                        [W.dynamic([], eob, [1]), W.fixed(b"x", final=1)], zd))
    # a 10-bit code next to 11-bit ones and an 8-bit next to 9-bit ones, on few symbols
    for lm, dm in [(11, 9), (10, 8)]:
        lit = [0] * 286
        for s, ln in zip([65, 66, 67, 256, 257, 280, 285] + list(range(100, 200)),
                         W.spine_lens(7 + 100, lm)):
            lit[s] = ln
        dist = [0] * 30
        for s, ln in zip([0, 3, 9, 17, 21, 29, 1, 2, 4, 5, 6, 7, 8], W.spine_lens(13, dm)):
            dist[s] = ln
        cases.append(_dyn("codes of %d next to %d bits, distances %d next to %d" % (lm - 1, lm, dm - 1, dm),
                          lit, dist, zd, rng))
    return [Group("code shapes", zd, cases)]


def _rle_span(blk, sym, count):
    """Expanded positions [p, p + count) of the first RLE item (sym, count), or None."""
    p = 0
    for r in blk["rle"]:
        if not isinstance(r, int) and r == (sym, count):
            return p, p + count
        p += 1 if isinstance(r, int) else r[1]
    return None


def family_dyn_headers():
    zd, rng, cases = dict32k(), _rng(2), []
    cases.append(_dyn("HLIT 257, HDIST 2", _lit_code(range(40, 90), n=257), [1, 1], zd, rng))
    lit = _lit_code(list(range(0, 256, 3)) + [285])
    assert len(lit) == 286 and lit[285]
    cases.append(_dyn("HLIT 286, HDIST 1", lit, [1], zd, rng))
    cases.append(_dyn("HLIT 286, HDIST 30", lit, W.spine_lens(30, 7), zd, rng))
    zeros = W.dynamic([], [0] * 286, [0], final=1)
    W.dynamic_header(zeros)
    assert zeros["hclen"] == 4
    cases.append(_invalid("HCLEN 4: only zero lengths, no end-of-block", [zeros], zd))
    lit8 = [0] + [8] * 256
    b = W.dynamic(tokens_using(lit8, [0], rng), lit8, [0], final=1)
    W.dynamic_header(b)
    assert b["hclen"] == 5
    cases.append(_valid("HCLEN 5: 256 codes of length 8", [b], zd))
    lit = [0] * 286
    for s, ln in zip(list(range(97, 112)) + [256], W.spine_lens(16, 15)):
        lit[s] = ln
    b = W.dynamic(tokens_using(lit, [0], rng), lit, [0], final=1)
    W.dynamic_header(b)
    assert b["hclen"] == 19 and b["cl_lens"][15] and b["cl_lens"][1]
    cases.append(_valid("HCLEN 19: code lengths 1 to 15", [b], zd))
    lit = _lit_code(range(48, 58))
    cases.append(_dyn("HCLEN 19 written with trailing zero lengths", lit, [0], zd, rng, hclen=19))
    # repeat codes at their minimum and maximum counts
    for sym, count in [(16, 3), (16, 6), (17, 3), (17, 10), (18, 11), (18, 138)]:
        lit = [0] * 286
        if sym == 16:
            lit[100:101 + count] = [8] * (count + 1)
        else:
            lit[100] = lit[101 + count] = 8
        lit[256] = 9
        W.fill_complete(lit, range(65, 91))
        b = W.dynamic(tokens_using(lit, [1, 1], rng), lit, [1, 1], final=1)
        W.dynamic_header(b)
        assert _rle_span(b, sym, count), (sym, count)
        cases.append(_valid("repeat %d x %d" % (sym, count), [b], zd))
    # a 16 that crosses from the literal/length lengths into the distance lengths
    lit = [0] * 286
    lit[284] = lit[285] = 6
    lit[256] = 7
    W.fill_complete(lit, range(65, 91))
    dist = [0] * 30
    dist[0:5] = [6] * 5
    W.fill_complete(dist, range(10, 30))
    b = W.dynamic(tokens_using(lit, dist, rng), lit, dist, final=1)
    W.dynamic_header(b)
    span = _rle_span(b, 16, 6)
    assert span and span[0] < 286 < span[1], span
    cases.append(_valid("repeat 16 across HLIT into the distance lengths", [b], zd))
    for sym, n_nonzero in [(17, 25), (18, 10)]:
        dist = W.balanced_lens(n_nonzero) + [0] * (30 - n_nonzero)
        b = W.dynamic(tokens_using(lit, dist, rng), lit, dist, final=1)
        W.dynamic_header(b)
        assert b["rle"][-1] == (sym, 30 - n_nonzero)
        cases.append(_valid("repeat %d x %d ends the vector" % (sym, 30 - n_nonzero), [b], zd))
    return [Group("dynamic headers", zd, cases)]


def _fixed_match_case(name, prefix, match, zd=b"", valid=True, extra=b"tail"):
    """A stored block `prefix` (when not empty), then a fixed block: the match, then a few literals."""
    blocks = ([W.stored(prefix)] if prefix else []) + [W.fixed([match] + list(extra), final=1)]
    return (_valid if valid else _invalid)(name, blocks, zd)


def family_tokens():
    groups, rng = [], _rng(3)
    pre = _bytes(rng, 300)
    cases = [_fixed_match_case("length %d" % n, pre, (n, int(rng.integers(1, 300)))) for n in range(3, 259)]
    cases.append(_fixed_match_case("length 258 as 284 + 31", pre, (258, 100, 284)))
    cases.append(_fixed_match_case("length 258 as 284 + 31, overlapping", pre, (258, 3, 284)))
    win = _bytes(rng, 32768)
    for c in range(30):
        for d in sorted({_DIST_BASE[c], _DIST_BASE[c] + (1 << _DIST_EXTRA[c]) - 1}):
            cases.append(_fixed_match_case("distance %d (code %d)" % (d, c), win, (int(rng.integers(3, 259)), d)))
    for d in range(1, 41):
        cases.append(_valid("overlapping copy, distance %d, length 258" % d,
                            [W.fixed(list(_bytes(rng, d)) + [(258, d)] + list(b"end"), final=1)]))
    for p in (1, 7, 300):
        lits = list(_bytes(rng, p))
        cases.append(_valid("distance = position %d" % p, [W.fixed(lits + [(10, p)], final=1)]))
        cases.append(_invalid("distance = position %d + 1" % p, [W.fixed(lits + [(10, p + 1)], final=1)], out_len=p + 10))
    groups.append(Group("tokens, no dictionary", b"", cases))
    for n in (1, 2, 31, 32, 33, 32767, 32768):
        zd, cases = _bytes(rng, n), []
        for p in (0, 1, 5, 40):
            if p + n <= 32768:
                lits = list(_bytes(rng, p))
                cases.append(_valid("pos %d, distance = pos + dict_len" % p, [W.fixed(lits + [(258, p + n)], final=1)], zd))
            if p + n + 1 <= 32768:
                cases.append(_invalid("pos %d, distance = pos + dict_len + 1" % p,
                                      [W.fixed(list(_bytes(rng, p)) + [(258, p + n + 1)], final=1)], zd, out_len=p + 258))
        for k in range(8):
            toks = [(int(rng.integers(3, 259)), int(rng.integers(1, n + 1))) for _ in range(4)]
            cases.append(_valid("matches into the dictionary %d" % k, [W.fixed(toks, final=1)], zd))
        cases.append(_valid("overlapping copy from the dictionary", [W.fixed([(258, min(n, 3)), (258, 1)], final=1)], zd))
        groups.append(Group("tokens, %d-byte dictionary" % n, zd, cases))
    return groups


def _tiny_blocks(rng, n):
    blocks, out = [], 0
    for i in range(n):
        kind = int(rng.integers(0, 3))
        if kind == 0:
            data = _bytes(rng, int(rng.integers(0, 6)))
            blocks.append(W.stored(data))
            out += len(data)
            continue
        toks = []
        for _ in range(int(rng.integers(0, 5))):
            if out and rng.random() < 0.4:
                toks.append((int(rng.integers(3, 259)), int(rng.integers(1, min(out, 32768) + 1))))
                out += toks[-1][0]
            else:
                toks.append(int(rng.integers(0, 256)))
                out += 1
        if kind == 1:
            blocks.append(W.fixed(toks))
        else:
            lsyms = {t for t in toks if isinstance(t, int)} | {W._len_sym(t[0]) for t in toks if not isinstance(t, int)}
            dsyms = sorted({W._dist_sym(t[1]) for t in toks if not isinstance(t, int)})
            dist = [0] * 30
            for s, ln in zip(dsyms, W.balanced_lens(len(dsyms)) if dsyms else []):
                dist[s] = ln
            blocks.append(W.dynamic(toks, _lit_code(lsyms), dist[:max(dsyms) + 1] if dsyms else [0]))
    blocks[-1]["final"] = 1
    return blocks


def family_blocks():
    rng, cases = _rng(4), []
    for n in (0, 1, 65535):
        cases.append(_valid("stored block of %d bytes" % n, [W.stored(_bytes(rng, n), final=1)]))
    cases.append(_valid("two stored blocks of 65535 bytes", [W.stored(_bytes(rng, 65535)), W.stored(_bytes(rng, 65535), final=1)]))
    for phase in range(8):
        b9 = (phase - 2) % 8   # 3 header bits + 5 eight-bit + b9 nine-bit literals + 7 end-of-block bits
        toks = list(b"abcde") + [200] * b9
        blocks = [W.fixed(toks), W.stored(_bytes(rng, 20), final=1)]
        assert (3 + 8 * 5 + 9 * b9 + 7) % 8 == phase
        cases.append(_valid("stored block at bit phase %d" % phase, blocks))
        blocks = [W.fixed(toks), W.stored(_bytes(rng, 3)), W.fixed([(5, 2), 7, 8], final=1)]
        cases.append(_valid("stored block at bit phase %d, then a fixed block" % phase, blocks))
    toks = list(_bytes(rng, 40)) + [(int(rng.integers(3, 259)), int(rng.integers(1, 41))) for _ in range(30)]
    cases.append(_valid("fixed block", [W.fixed(toks, final=1)]))
    cases.append(_valid("three fixed blocks", [W.fixed(toks[:20]), W.fixed(toks[20:40]), W.fixed(toks[40:], final=1)]))
    cases.append(_valid("empty fixed block", [W.fixed([], final=1)]))
    for seed in range(3):
        cases.append(_valid("2000 tiny mixed blocks, seed %d" % seed, _tiny_blocks(_rng(40 + seed), 2000)))
    cases.append(_invalid("a block after the final one", [W.fixed(b"one", final=1), W.fixed(b"two", final=1)]))
    cases.append(_invalid("no final block", [W.fixed(b"one"), W.fixed(b"two")]))
    return [Group("blocks", b"", cases)]


def _text(rng, n):
    words = [bytes(rng.integers(97, 123, int(rng.integers(2, 9)), dtype=np.uint8)) + b" " for _ in range(300)]
    out = bytearray()
    while len(out) < n:
        out += words[int(rng.integers(0, len(words)))]
    return bytes(out[:n])


def _zcase(name, data, zd=b"", level=6, valid=True, out_len=None, status=None, edit=None):
    c = zlib.compressobj(level, zlib.DEFLATED, 15, 8, zlib.Z_DEFAULT_STRATEGY, **({"zdict": zd} if zd else {}))
    s = c.compress(data) + c.flush()
    if edit:
        s = edit(bytearray(s))
    n = len(data) if out_len is None else out_len
    return Case(name, s, n, valid, data if valid else None, status)


def family_header_trailer():
    rng = _rng(5)
    data = _text(rng, 3000)
    blocks = [W.fixed(list(data[:200]) + [(100, 50)], final=1)]
    good, raw = W.zlib_stream(blocks)
    cases = []
    for cinfo in range(9):
        cmf, flg = W.header(cmf=(cinfo << 4) | 8)
        cases.append((_valid if cinfo <= 7 else _invalid)("CINFO %d" % cinfo, blocks, cmf=cmf, flg=flg))
    cmf, flg = W.header(cmf=0x08)
    far = [W.stored(_bytes(rng, 32768)), W.fixed([(258, 32768)], final=1)]
    cases.append(_valid("CINFO 0 and a distance of 32768", far, cmf=cmf, flg=flg))
    for cm in (0, 7, 9, 15):
        cmf, flg = W.header(cmf=0x70 | cm)
        cases.append(_invalid("compression method %d" % cm, blocks, cmf=cmf, flg=flg))
    for lv in range(4):
        cmf, flg = W.header(flevel=lv)
        cases.append(_valid("FLEVEL %d" % lv, blocks, cmf=cmf, flg=flg))
    cmf, flg = W.header(fcheck_ok=False)
    cases.append(_invalid("wrong FCHECK", blocks, cmf=cmf, flg=flg))
    cmf, flg = W.header(fdict=True)
    cases.append(_invalid("FDICT without a dictionary", blocks, cmf=cmf, flg=flg, dictid=zlib.adler32(b"x")))
    for i in range(4):
        for delta in (1, -1):
            t = bytearray(good)
            t[len(t) - 4 + i] = (t[len(t) - 4 + i] + delta) & 0xFF
            cases.append(Case("trailer byte %d %+d" % (i, delta), t, len(raw), False))
    for k in range(1, 5):
        cases.append(Case("trailer cut by %d byte(s)" % k, good[:-k], len(raw), False))
    cases.append(Case("one byte after the trailer", good + b"\0", len(raw), False))
    cases.append(Case("expected length - 1", good, len(raw) - 1, False))
    cases.append(Case("expected length + 1", good, len(raw) + 1, False, status=5))
    cases.append(Case("expected length 0", good, 0, False))
    big = _text(rng, 270000)
    big = big[:60000] + _bytes(rng, 20000) + big[80000:]
    for n in (131071, 131072, 131073, 4096 * 32 * 2 + 1):
        for level in (0, 6):
            cases.append(_zcase("%d bytes, level %d" % (n, level), big[:n], level=level))
    cases.append(_zcase("empty output", b""))
    nodict = Group("header and trailer, no dictionary", b"", cases)

    zd = _text(rng, 2000)
    cases = [_zcase("with the dictionary", data, zd), _zcase("with the dictionary, level 9", data, zd, level=9)]
    cases.append(_zcase("a dictionary without FDICT", data, valid=False))
    for delta in (1, -1):
        def edit(s, delta=delta):
            s[2:6] = ((int.from_bytes(s[2:6], "big") + delta) & 0xFFFFFFFF).to_bytes(4, "big")
            return bytes(s)
        cases.append(_zcase("DICTID %+d" % delta, data, zd, valid=False, status=1, edit=edit))
    cases.append(_zcase("expected length + 1, with the dictionary", data, zd, valid=False, out_len=len(data) + 1, status=5))
    cases.append(_zcase("expected length - 1, with the dictionary", data, zd, valid=False, out_len=len(data) - 1))
    withdict = Group("header and trailer, with a dictionary", zd, cases)
    return [nodict, withdict]


def family_invalid():
    zd, rng, cases = dict32k(), _rng(6), []
    lit = W.spine_lens(286, 12)
    dist = W.spine_lens(30, 10)
    toks = tokens_using(lit, dist, rng)
    cases.append(_dyn("valid reference block", lit, dist, zd, rng, tokens=toks))
    over = list(lit)
    over[over.index(12)] = 11
    cases.append(_dyn("over-subscribed literal/length code", over, dist, zd, rng, valid=False, tokens=toks))
    over = list(dist)
    over[over.index(10)] = 9
    cases.append(_dyn("over-subscribed distance code", lit, over, zd, rng, valid=False, tokens=toks))
    inc = list(lit)
    inc[inc.index(12)] = 13
    cases.append(_dyn("incomplete literal/length code", inc, dist, zd, rng, valid=False, tokens=toks))
    inc = list(dist)
    inc[inc.index(10)] = 11
    cases.append(_dyn("incomplete distance code", lit, inc, zd, rng, valid=False, tokens=toks))
    cases.append(_dyn("three distance codes of length 2", lit, [2, 2, 2], zd, rng, valid=False,
                      tokens=[97, (5, 1), (9, 2), (20, 3)]))
    blk = W.dynamic_header(W.dynamic(toks, lit, dist, final=1))
    cl = list(blk["cl_lens"])
    used = [s for s in range(19) if cl[s]]
    cl2 = list(cl)
    cl2[next(s for s in range(19) if not cl[s])] = min(cl[s] for s in used)   # one code too many
    cases.append(_dyn("over-subscribed code-length code", lit, dist, zd, rng, valid=False, tokens=toks, cl_lens=cl2))
    cl2 = list(cl)
    cl2[max(used, key=lambda s: cl[s])] += 1   # one leaf moves down a level: incomplete
    cases.append(_dyn("incomplete code-length code", lit, dist, zd, rng, valid=False, tokens=toks, cl_lens=cl2))
    cases.append(_dyn("code-length code with no codes", lit, dist, zd, rng, valid=False, tokens=toks, cl_lens=[0] * 19))
    for L in range(2, 16):
        eob = [0] * 257
        eob[256] = L
        cases.append(_dyn("end-of-block alone at length %d" % L, eob, [0], zd, rng, valid=False, tokens=[]))
    base = _lit_code(list(range(97, 123)) + [257, 266, 285])
    for L in range(2, 16):
        d = [0] * 6
        d[5] = L
        cases.append(_dyn("single distance code of length %d" % L, base, d, zd, rng, valid=False,
                          tokens=[97, (3, 7), 98, (258, 8)]))
    eob = [0] * 257
    eob[256] = 1
    cases.append(_dyn("end-of-block alone at length 1, then the unused code 1", eob, [0], zd, rng, valid=False,
                      tokens=[("bits", 1, 1)]))
    cases.append(_dyn("single distance code of length 1, then the unused code 1", base, [1], zd, rng, valid=False,
                      tokens=[97, ("len", 4), ("bits", 1, 1), 98]))
    cases.append(_dyn("a match with no distance code", base, [0], zd, rng, valid=False,
                      tokens=[97, ("len", 4), ("bits", 0, 5), 98]))
    noeob = list(lit)
    noeob[256] = 0
    cases.append(_dyn("no end-of-block code", noeob, dist, zd, rng, valid=False, tokens=[t for t in toks if t != 256]))
    rle = W.rle_encode(lit + dist)
    cases.append(_dyn("repeat 16 first", lit, dist, zd, rng, valid=False, tokens=toks, rle=[(16, 3)] + rle[1:]))
    over = rle[:-1] + [(18, 138)]
    cases.append(_dyn("RLE overruns HLIT + HDIST", lit, dist, zd, rng, valid=False, tokens=toks, rle=over))
    dz = W.balanced_lens(27) + [0, 0, 0]
    rle = W.rle_encode(lit + dz)
    assert rle[-1] == (17, 3)
    cases.append(_dyn("RLE overruns by one", lit, dz, zd, rng, valid=False, tokens=toks[:5], rle=rle[:-1] + [(17, 4)]))
    for hlit, hdist in [(287, 30), (288, 30), (286, 31), (286, 32)]:
        cases.append(_dyn("HLIT %d HDIST %d" % (hlit, hdist), lit, dist, zd, rng, valid=False, tokens=toks,
                          hlit=hlit, hdist=hdist))
    for s in (286, 287):
        cases.append(_invalid("literal/length symbol %d in a fixed block" % s, [W.fixed([97, ("sym", s), 98], final=1)], zd,
                              out_len=2))
    for d in (30, 31):
        cases.append(_invalid("distance symbol %d in a fixed block" % d, [W.fixed([97, ("dsym", 3, d), 98], final=1)], zd,
                              out_len=5))
    cases.append(_invalid("block type 3", [{"final": 1, "type": 3, "tokens": []}], zd))
    cases.append(_invalid("block type 3 after a stored block", [W.stored(b"abc"), {"final": 1, "type": 3, "tokens": []}], zd,
                          out_len=3))
    for ln, nln in [(5, 5), (5, 0xFFFF ^ 4), (0, 0), (0xFFFF, 0xFFFF)]:
        b = W.stored(b"hello", final=1)
        b["len_nlen"] = (ln, nln)
        cases.append(_invalid("stored LEN %d NLEN %d" % (ln, nln), [b], zd))
    return [Group("invalid structure", zd, cases)]


def damaged_sources():
    """Three small valid streams: stored, fixed, and dynamic with a dictionary: (name, stream, raw, zd)."""
    rng = _rng(7)
    s1, r1 = W.zlib_stream([W.stored(b"stored block, twenty", final=1)])
    s2, r2 = W.zlib_stream([W.fixed(list(b"fixed code: abcabcabc") + [(20, 3), 33, (7, 21)], final=1)])
    zd = _text(rng, 500)
    lit = _lit_code(list(range(97, 110)) + [258, 262, 270])
    dist = [0, 2, 2, 0, 0, 0, 0, 0, 2, 0, 0, 0, 0, 0, 0, 0, 2]   # distance codes 1, 2, 8 and 16
    toks = [97, (4, 2), 98, (23, 300), 99, (8, 18), 100, (8, 3), 101, (25, 2)]
    s3, r3 = W.zlib_stream([W.dynamic(toks, lit, dist, final=1)], zd)
    return [("stored", s1, r1, b""), ("fixed", s2, r2, b""), ("dynamic with a dictionary", s3, r3, zd)]


def family_damaged():
    groups = {}
    for name, s, raw, zd in damaged_sources():
        cases = groups.setdefault(zd, [])
        cases.append(Case("%s: intact" % name, s, len(raw), True, raw))
        for n in range(len(s)):
            cases.append(Case("%s: cut to %d of %d bytes" % (name, n, len(s)), s[:n], len(raw), None))
        for i in range(len(s)):
            t = bytearray(s)
            t[i] ^= 1 << (i % 8)
            cases.append(Case("%s: bit %d of byte %d flipped" % (name, i % 8, i), t, len(raw), None))
    return [Group("damaged, %s" % ("no dictionary" if not zd else "with a dictionary"), zd, c) for zd, c in groups.items()]


FAMILIES = {
    "code_shapes": family_code_shapes,
    "dyn_headers": family_dyn_headers,
    "tokens": family_tokens,
    "blocks": family_blocks,
    "header_trailer": family_header_trailer,
    "invalid": family_invalid,
    "damaged": family_damaged,
}
