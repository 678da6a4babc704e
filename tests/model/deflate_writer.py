"""The inverse of `inflate_tokens.read_zlib`: `write_zlib(s)` turns the dict the reader returns back into the bytes of
the stream, canonical codes from the code lengths (RFC 1951 section 3.2.2), zero padding bits as zlib writes them.
TEST INFRASTRUCTURE: it writes what the reader (and zlib) reject just as readily, because the decoder's tests need
malformed streams of every kind.  Nothing is checked; these fields override what a valid stream would hold:

  stream  'trailer' (raw bytes instead of the big-endian 'adler'), 'tail' (bytes after the trailer); 'dictid' is
          written iff it is not None, whatever FDICT says
  block   'len_nlen' (LEN, NLEN of a stored block); type 3 writes the three header bits and nothing else;
          'hlit' / 'hdist' / 'hclen' / 'cl_lens' / 'rle' are written as given (lengths that over-subscribe or leave
          the code incomplete, a 16 first, an RLE that overruns HLIT + HDIST); 'no_eob' leaves out end-of-block
  token   an int is a literal, (length, distance) a match coded the usual way (258 as symbol 285),
          (length, distance, lsym) a match whose length is coded with symbol lsym (284 + 31 extra bits for 258),
          ('sym', s) a bare literal/length symbol (286, 287), ('dsym', length, d) a length followed by the bare
          distance symbol d (30, 31), ('len', length) a length with no distance after it, ('bits', v, n) n raw
          bits (a bit pattern outside an incomplete code)

A dynamic block only needs 'lit_lens', 'dist_lens' and 'tokens': the header fields the reader returns are derived
when missing (HLIT / HDIST from the vectors' lengths, a greedy RLE as zlib's, a complete code-length code)."""
import zlib

from tests.model.inflate_tokens import (_CL_ORDER, _DIST_BASE, _DIST_EXTRA, _FIXED_DIST, _FIXED_LIT, _LEN_BASE,
                                        _LEN_EXTRA, _rev, replay)


class BitWriter:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def put(self, v, nb):   # LSB first
        self.acc |= (v & ((1 << nb) - 1)) << self.n
        self.n += nb
        while self.n >= 8:
            self.out.append(self.acc & 0xFF)
            self.acc >>= 8
            self.n -= 8

    def code(self, c, ln):   # Huffman codes go MSB first
        self.put(_rev(c, ln), ln)

    def align(self):
        if self.n:
            self.put(0, 8 - self.n)

    def raw(self, b):
        assert self.n == 0
        self.out += b


def canonical_codes(lens):
    """symbol -> code of the canonical code of `lens` (RFC 1951 3.2.2; over-subscribed lengths give codes anyway)."""
    bl = [0] * 16
    for ln in lens:
        if ln:
            bl[ln] += 1
    code, nxt = 0, [0] * 16
    for b in range(1, 16):
        code = (code + bl[b - 1]) << 1
        nxt[b] = code
    codes = {}
    for s, ln in enumerate(lens):
        if ln:
            codes[s] = nxt[ln]
            nxt[ln] += 1
    return codes


def _len_sym(ln):
    if ln == 258:
        return 285
    return max(i for i in range(29) if _LEN_BASE[i] <= ln) + 257


def _dist_sym(d):
    return max(i for i in range(30) if _DIST_BASE[i] <= d)


def rle_encode(lens):
    """Greedy code-length RLE, as zlib writes it: 18 / 17 for zero runs, a length and 16s for other runs."""
    out, i = [], 0
    while i < len(lens):
        v, r = lens[i], 1
        while i + r < len(lens) and lens[i + r] == v:
            r += 1
        i += r
        if v == 0:
            while r >= 11:
                k = min(r, 138)
                out.append((18, k))
                r -= k
            if r >= 3:
                out.append((17, r))
                r = 0
            out += [0] * r
        else:
            out.append(v)
            r -= 1
            while r >= 3:
                k = min(r, 6)
                out.append((16, k))
                r -= k
            out += [v] * r
    return out


def balanced_lens(k):
    """Lengths of a complete code of k >= 2 symbols as balanced as it gets (k = 1: a single code of length 1)."""
    if k == 1:
        return [1]
    L = (k - 1).bit_length()
    a = (1 << L) - k   # this many symbols one bit shorter
    return [L - 1] * a + [L] * (k - a)


def spine_lens(n, maxlen):
    """Lengths of a Kraft-complete code of n symbols whose longest code has exactly `maxlen` bits: a spine of one code
    per length D+1 .. maxlen-1 and two of maxlen fills one node of depth D, the other 2^D - 1 nodes hold the rest at
    depth D and D+1.  So a code of maxlen-1 bits sits next to the maxlen-bit ones in canonical order."""
    for D in range(1, maxlen):
        q, r = (1 << D) - 1, n - (maxlen - D + 1)
        if q <= r <= 2 * q:
            x = r - q   # nodes split into two
            lens = [D] * (q - x) + [D + 1] * (2 * x) + list(range(D + 1, maxlen)) + [maxlen, maxlen]
            assert len(lens) == n and sum(2 ** (15 - v) for v in lens) == 2 ** 15
            return lens
    raise ValueError("no spine code of %d symbols with max length %d" % (n, maxlen))


def kraft(lens):
    """Code space used, in units of 2^-15: 2^15 for a complete code."""
    return sum(1 << (15 - v) for v in lens if v)


def fill_complete(lens, free):
    """Completes `lens` in place with codes at positions `free` (in order): one code per set bit of the slack."""
    slack = (1 << 15) - kraft(lens)
    assert slack >= 0
    free = iter(free)
    for b in range(15):
        if slack >> b & 1:
            p = next(free)
            assert lens[p] == 0
            lens[p] = 15 - b
    return lens


def cl_code(rle):
    """A complete code-length code over the RLE's symbols (two symbols at least: 0 is added when alone)."""
    used = sorted({t if isinstance(t, int) else t[0] for t in rle})
    if len(used) == 1:
        used = sorted(set(used) | {0 if used[0] else 1})
    lens = [0] * 19
    for s, ln in zip(used, balanced_lens(len(used))):
        lens[s] = ln
    return lens


def _hclen(cl):
    n = 19
    while n > 4 and cl[_CL_ORDER[n - 1]] == 0:
        n -= 1
    return n


def dynamic_header(blk):
    """Fills in the header fields of a dynamic block that are missing (see the module's docstring)."""
    lit, dist = blk["lit_lens"], blk["dist_lens"]
    blk.setdefault("hlit", len(lit))
    blk.setdefault("hdist", len(dist))
    blk.setdefault("rle", rle_encode(list(lit) + list(dist)))
    blk.setdefault("cl_lens", cl_code(blk["rle"]))
    blk.setdefault("hclen", _hclen(blk["cl_lens"]))
    return blk


def _write_tokens(bw, toks, lit_lens, dist_lens, no_eob):
    lc, dc = canonical_codes(lit_lens), canonical_codes(dist_lens)

    def sym(codes, lens, s):
        bw.code(codes.get(s, 0), lens[s] if s < len(lens) and lens[s] else 1)

    def match(ln, lsym):
        sym(lc, lit_lens, lsym)
        bw.put(ln - _LEN_BASE[lsym - 257], _LEN_EXTRA[lsym - 257])

    for t in toks:
        if isinstance(t, int):
            sym(lc, lit_lens, t)
        elif t[0] == "sym":
            sym(lc, lit_lens, t[1])
        elif t[0] == "dsym":
            match(t[1], _len_sym(t[1]))
            sym(dc, dist_lens, t[2])
        elif t[0] == "len":
            match(t[1], _len_sym(t[1]))
        elif t[0] == "bits":
            bw.put(t[1], t[2])
        else:
            ln, d = t[0], t[1]
            match(ln, t[2] if len(t) > 2 else _len_sym(ln))
            ds = _dist_sym(d)
            sym(dc, dist_lens, ds)
            bw.put(d - _DIST_BASE[ds], _DIST_EXTRA[ds])
    if not no_eob:
        sym(lc, lit_lens, 256)


def write_block(bw, blk):
    bw.put(blk["final"], 1)
    bw.put(blk["type"], 2)
    t = blk["type"]
    if t == 0:
        bw.align()
        data = blk["stored"]
        ln, nln = blk.get("len_nlen", (len(data), len(data) ^ 0xFFFF))
        bw.put(ln, 16)
        bw.put(nln, 16)
        bw.raw(data)
    elif t == 1:
        _write_tokens(bw, blk["tokens"], _FIXED_LIT, _FIXED_DIST + [5, 5], blk.get("no_eob"))
    elif t == 2:
        dynamic_header(blk)
        bw.put(blk["hlit"] - 257, 5)
        bw.put(blk["hdist"] - 1, 5)
        bw.put(blk["hclen"] - 4, 4)
        cl = blk["cl_lens"]
        for i in range(blk["hclen"]):
            bw.put(cl[_CL_ORDER[i]], 3)
        cc = canonical_codes(cl)
        for r in blk["rle"]:
            s = r if isinstance(r, int) else r[0]
            bw.code(cc.get(s, 0), cl[s] or 1)
            if not isinstance(r, int):
                bw.put(r[1] - (11 if s == 18 else 3), {16: 2, 17: 3, 18: 7}[s])
        _write_tokens(bw, blk["tokens"], blk["lit_lens"], blk["dist_lens"], blk.get("no_eob"))


def write_deflate(blocks):
    bw = BitWriter()
    for b in blocks:
        write_block(bw, b)
    bw.align()
    return bytes(bw.out)


def write_zlib(s):
    """The bytes of the stream `s` (a dict as `read_zlib` returns it, with the overrides of the module docstring)."""
    out = bytearray([s["cmf"], s["flg"]])
    if s.get("dictid") is not None:
        out += s["dictid"].to_bytes(4, "big")
    out += write_deflate(s["blocks"])
    out += s["trailer"] if "trailer" in s else s["adler"].to_bytes(4, "big")
    return bytes(out + s.get("tail", b""))


def header(cmf=0x78, flevel=2, fdict=False, fcheck_ok=True):
    """(CMF, FLG) with a correct FCHECK (or one off by one)."""
    flg = (flevel << 6) | (0x20 if fdict else 0)
    flg |= (31 - (cmf * 256 + flg) % 31) % 31
    if not fcheck_ok:
        flg ^= 1   # bit 0 belongs to FCHECK: the header moves by one, off a multiple of 31
    return cmf, flg


def stored(data, final=0):
    return {"final": final, "type": 0, "stored": bytes(data), "tokens": list(bytes(data))}


def fixed(tokens, final=0, **kw):
    return dict({"final": final, "type": 1, "tokens": list(tokens)}, **kw)


def dynamic(tokens, lit_lens, dist_lens, final=0, **kw):
    return dict({"final": final, "type": 2, "tokens": list(tokens), "lit_lens": list(lit_lens),
                 "dist_lens": list(dist_lens)}, **kw)


def output(blocks, zd=b""):
    """The bytes the tokens of `blocks` stand for; ValueError when a token has no meaning (a bare symbol, a distance
    before the window)."""
    norm = []
    for b in blocks:
        toks = []
        for t in b.get("tokens", []):
            if not isinstance(t, int) and (isinstance(t[0], str) or len(t) != 2 and len(t) != 3):
                raise ValueError("token %r stands for no bytes" % (t,))
            toks.append(t if isinstance(t, int) else (t[0], t[1]))
        norm.append({"tokens": toks})
    return replay(norm, zd)


def zlib_stream(blocks, zd=b"", **kw):
    """(stream, raw bytes) of `blocks` with a correct header, DICTID iff zd, and Adler-32 trailer; keyword arguments
    override fields of the stream dict ('trailer', 'tail', 'dictid', 'cmf', 'flg', 'adler', ...).  raw is None when
    the tokens stand for no bytes (the Adler-32 is 0 then, unless given)."""
    try:
        raw = output(blocks, zd)
    except ValueError:
        raw = None
    cmf, flg = header(fdict=bool(zd))
    s = {"cmf": cmf, "flg": flg, "dictid": zlib.adler32(zd) if zd else None, "blocks": blocks,
         "adler": zlib.adler32(raw) if raw is not None else 0}
    s.update(kw)
    return write_zlib(s), raw
