"""A small pure-Python RFC 1950 / RFC 1951 reader that keeps the structure of a stream: header and DICTID, per block its
type, HLIT / HDIST / HCLEN, the code lengths and the tokens (a literal byte, or a (length, distance) pair), and the
trailer.  TEST INFRASTRUCTURE: when two encoders disagree on a stream, `first_difference` names the first differing
header field, code length or token instead of a byte offset inside a bit string.  Malformed input raises ValueError;
it is not a validating inflater (stock zlib is that)."""

_LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
_LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
_DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
              4097, 6145, 8193, 12289, 16385, 24577]
_DIST_EXTRA = [0, 0, 0, 0] + [i // 2 for i in range(2, 28)]
_CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
_FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
_FIXED_DIST = [5] * 30


class _Bits:
    def __init__(self, data, pos=0):
        self.d = bytes(data) + b"\0\0\0\0"
        self.n = len(data)
        self.pos = pos * 8   # bit position

    def peek(self, nb):   # nb <= 24
        i = self.pos >> 3
        return (int.from_bytes(self.d[i:i + 4], "little") >> (self.pos & 7)) & ((1 << nb) - 1)

    def get(self, nb):
        if nb == 0:
            return 0
        v = self.peek(nb)
        self.skip(nb)
        return v

    def skip(self, nb):
        self.pos += nb
        if self.pos > 8 * self.n:
            raise ValueError("stream ends inside a block")

    def align(self):
        self.pos = (self.pos + 7) & ~7


def _rev(v, n):
    r = 0
    for _ in range(n):
        r = (r << 1) | (v & 1)
        v >>= 1
    return r


class _Decoder:
    """Canonical Huffman decoding by a table of all 15-bit LSB-first prefixes."""

    def __init__(self, lens):
        if not any(lens):
            self.table = None
            return
        self.maxb = max(lens)
        bl = [0] * 16
        for ln in lens:
            if ln:
                bl[ln] += 1
        code, nxt = 0, [0] * 16
        for b in range(1, 16):
            code = (code + bl[b - 1]) << 1
            nxt[b] = code
        self.table = [None] * (1 << self.maxb)
        for s, ln in enumerate(lens):
            if not ln:
                continue
            c = _rev(nxt[ln], ln)
            nxt[ln] += 1
            for k in range(c, 1 << self.maxb, 1 << ln):
                self.table[k] = (s, ln)

    def sym(self, br):
        if self.table is None:
            raise ValueError("symbol read from an empty code")
        e = self.table[br.peek(self.maxb)]
        if e is None:
            raise ValueError("bit pattern outside the code (incomplete code)")
        br.skip(e[1])
        return e[0]


def _coded_block(br, blk, lit_lens, dist_lens):
    lit, dst = _Decoder(lit_lens), _Decoder(dist_lens)
    toks = blk["tokens"]
    while True:
        s = lit.sym(br)
        if s < 256:
            toks.append(s)
        elif s == 256:
            return
        else:
            s -= 257
            if s >= 29:
                raise ValueError("length symbol %d" % (s + 257))
            ln = _LEN_BASE[s] + br.get(_LEN_EXTRA[s])
            d = dst.sym(br)
            if d >= 30:
                raise ValueError("distance symbol %d" % d)
            toks.append((ln, _DIST_BASE[d] + br.get(_DIST_EXTRA[d])))


def read_deflate(data, pos=0):
    """Blocks of the raw DEFLATE stream that starts at byte `pos`; returns (blocks, byte position after the last one)."""
    br = _Bits(data, pos)
    blocks = []
    while True:
        final, btype = br.get(1), br.get(2)
        blk = {"final": final, "type": btype, "tokens": []}
        blocks.append(blk)
        if btype == 0:
            br.align()
            ln, nln = br.get(16), br.get(16)
            if ln ^ nln != 0xFFFF:
                raise ValueError("stored block LEN / NLEN mismatch")
            i = br.pos >> 3
            if i + ln > br.n:
                raise ValueError("stored block runs past the end")
            blk["stored"] = bytes(br.d[i:i + ln])
            blk["tokens"].extend(blk["stored"])
            br.pos += 8 * ln
        elif btype == 1:
            blk["lit_lens"], blk["dist_lens"] = list(_FIXED_LIT), list(_FIXED_DIST)
            _coded_block(br, blk, blk["lit_lens"], blk["dist_lens"])
        elif btype == 2:
            hlit, hdist, hclen = br.get(5) + 257, br.get(5) + 1, br.get(4) + 4
            cl = [0] * 19
            for i in range(hclen):
                cl[_CL_ORDER[i]] = br.get(3)
            cld = _Decoder(cl)
            lens, rle = [], []
            while len(lens) < hlit + hdist:
                s = cld.sym(br)
                if s < 16:
                    rle.append(s)
                    lens.append(s)
                elif s == 16:
                    if not lens:
                        raise ValueError("repeat code 16 with no previous length")
                    r = 3 + br.get(2)
                    rle.append((16, r))
                    lens.extend([lens[-1]] * r)
                else:
                    r = (3 + br.get(3)) if s == 17 else (11 + br.get(7))
                    rle.append((s, r))
                    lens.extend([0] * r)
            if len(lens) != hlit + hdist:
                raise ValueError("code lengths overrun HLIT + HDIST")
            blk.update(hlit=hlit, hdist=hdist, hclen=hclen, cl_lens=cl, rle=rle, lit_lens=lens[:hlit],
                       dist_lens=lens[hlit:])
            _coded_block(br, blk, blk["lit_lens"], blk["dist_lens"])
        else:
            raise ValueError("block type 3")
        if final:
            br.align()
            return blocks, br.pos >> 3


def read_zlib(data):
    """{'cmf', 'flg', 'dictid' (or None), 'blocks', 'adler', 'end'} of one RFC 1950 stream."""
    data = bytes(data)
    if len(data) < 6:
        raise ValueError("shorter than a zlib stream")
    cmf, flg = data[0], data[1]
    if (cmf * 256 + flg) % 31 or cmf & 15 != 8:
        raise ValueError("bad zlib header %02x %02x" % (cmf, flg))
    pos, dictid = 2, None
    if flg & 0x20:
        dictid = int.from_bytes(data[2:6], "big")
        pos = 6
    blocks, end = read_deflate(data, pos)
    if end + 4 > len(data):
        raise ValueError("stream ends inside the trailer")
    return {"cmf": cmf, "flg": flg, "dictid": dictid, "blocks": blocks, "adler": int.from_bytes(data[end:end + 4], "big"),
            "end": end + 4}


def replay(blocks, zdict=b""):
    """The bytes the tokens of `blocks` stand for (distances may reach into the preset dictionary)."""
    out = bytearray(zdict)
    base = len(out)
    for b in blocks:
        for t in b["tokens"]:
            if isinstance(t, int):
                out.append(t)
            else:
                ln, d = t
                if d > len(out) or d > 32768:
                    raise ValueError("distance %d reaches before the window" % d)
                s = len(out) - d
                for i in range(ln):   # overlapping copies repeat the bytes just written
                    out.append(out[s + i])
    return bytes(out[base:])


def _tok(t):
    return "literal %d" % t if isinstance(t, int) else "match length %d distance %d" % t


def first_difference(a, b):
    """Where zlib streams a and b (bytes) first differ, in stream terms; None when they are equal byte for byte."""
    a, b = bytes(a), bytes(b)
    if a == b:
        return None
    try:
        sa = read_zlib(a)
    except ValueError as e:
        return "first stream unreadable: %s" % e
    try:
        sb = read_zlib(b)
    except ValueError as e:
        return "second stream unreadable: %s" % e
    for f in ("cmf", "flg", "dictid"):
        if sa[f] != sb[f]:
            return "header %s: %r vs %r" % (f, sa[f], sb[f])
    pos = 0   # input position of the current token
    for k in range(max(len(sa["blocks"]), len(sb["blocks"]))):
        if k >= len(sa["blocks"]) or k >= len(sb["blocks"]):
            return "block count: %d vs %d" % (len(sa["blocks"]), len(sb["blocks"]))
        x, y = sa["blocks"][k], sb["blocks"][k]
        # the first differing token is usually the cause and the code lengths follow from it: both are named
        found, start = [], pos
        for i, (u, v) in enumerate(zip(x["tokens"], y["tokens"])):
            if u != v:
                found.append("token %d (input offset %d): %s vs %s" % (i, pos, _tok(u), _tok(v)))
                break
            pos += 1 if isinstance(u, int) else u[0]
        if not found and len(x["tokens"]) != len(y["tokens"]):
            found.append("%d vs %d tokens" % (len(x["tokens"]), len(y["tokens"])))
        for f in ("final", "type", "hlit", "hdist", "hclen"):
            if x.get(f) != y.get(f):
                found.append("%s %r vs %r" % (f, x.get(f), y.get(f)))
                break
        else:
            for f in ("lit_lens", "dist_lens", "cl_lens"):
                if x.get(f) != y.get(f):
                    i = next(i for i, (u, v) in enumerate(zip(x[f], y[f])) if u != v)
                    found.append("%s[%d] = %d vs %d" % (f, i, x[f][i], y[f][i]))
                    break
        if found:
            return "block %d (input offset %d): %s" % (k, start, "; ".join(found))
    if sa["adler"] != sb["adler"]:
        return "trailer Adler-32: %08x vs %08x" % (sa["adler"], sb["adler"])
    if len(a) != len(b):
        return "stream length %d vs %d with equal content" % (len(a), len(b))
    i = next(i for i in range(len(a)) if a[i] != b[i])
    return "equal structure, byte %d differs (padding bits?)" % i
