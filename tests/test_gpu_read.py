"""Random-access reads (hmse_read_open / hmse_read, archive.Reader): byte ranges of v1, v2 and v3 archives equal slices of
the input and the zlib-only reader's stats (tests/read_ref.py); every stored chunk and delta a batch needs is inflated /
applied once; a damaged chunk fails exactly the ranges that need it; damaged records fail the open; bad ranges fail the
call before anything is written; the kernel count does not depend on the batch; scratch follows the batch."""
import ctypes as C

import numpy as np
import pytest

from oracle import corpus
from tests import read_ref

pytestmark = pytest.mark.gpu


def _chunk_ends(ar):
    return np.cumsum(ar.pointers[:, 6:8].copy().view("<u2").reshape(-1).astype(np.int64) + 1)


def _positions(ar):
    return ar.pointers[:, 0:4].copy().view("<u4").reshape(-1).astype(np.int64) * 512 + ar.pointers[:, 4:6].copy().view("<u2").reshape(-1)


@pytest.fixture(scope="module")
def archives(ctx, corpus8):
    """kind -> (data, Archive, container bytes, file sizes or None), built on the device from corpus data with repeats."""
    import hmse_b200
    from hmse_b200 import archive
    zd = corpus.zdict()
    out = {}
    d1 = np.concatenate([corpus8[:3 << 20], corpus8[1 << 20:2 << 20], corpus8[:1 << 20]])
    ar = archive.build(hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(d1)), zd, ctx=ctx)
    out["v1"] = (d1, ar, ar.tobytes(), None)
    d2 = np.concatenate([corpus8[:6 << 20], corpus8[2 << 20:3 << 20]])
    ar = archive.build(hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(d2), l4=hmse_b200.SimConfig()), zd, ctx=ctx)
    assert ar.n_delta > 20
    out["v2"] = (d2, ar, ar.tobytes(), None)
    rng = np.random.default_rng(9)
    d3 = np.concatenate([corpus8[:2 << 20], corpus8[512 << 10:1 << 20]])
    sizes = rng.integers(0, 64 << 10, 60)
    sizes[rng.random(60) < 0.2] = 0
    sizes = np.concatenate([[0], sizes, [d3.size - int(sizes.sum())], [0]])
    assert sizes[-2] > 0
    ar = archive.build(hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(d3), files=sizes), zd, ctx=ctx)
    out["v3"] = (d3, ar, ar.tobytes(), sizes)
    return out


def _edge_ranges(rng, ends, raw):
    """lengths 0, 1, one chunk, many chunks, the whole stream; starts on the last byte of a chunk, ends on a cut."""
    starts = np.concatenate([[0], ends[:-1]])
    k = rng.integers(0, ends.size, 12)
    r = [(0, raw), (raw, 0), (0, 0), (raw - 1, 1), (0, 1), (int(ends[0]) - 1, 1)]
    for c in k:
        cs, ce = int(starts[c]), int(ends[c])
        r += [(cs, ce - cs), (ce - 1, 1), (ce - 1, 2 if ce < raw else 1), (cs, 0), (cs + (ce - cs) // 2, ce - cs - (ce - cs) // 2)]
        c2 = min(int(c) + int(rng.integers(2, 40)), ends.size - 1)
        r += [(cs, int(ends[c2]) - cs), (ce - 1, int(ends[c2]) - ce + 1)]
    return r


def _check(ctx, kind, archives, ranges, files=None):
    from hmse_b200 import archive
    data, ar, buf, sizes = archives[kind]
    rd = archive.Reader(ar, ctx)
    off = np.array([a for a, _ in ranges], dtype=np.uint64)
    ln = np.array([b for _, b in ranges], dtype=np.uint64)
    st, ost = {}, {}
    got, goff = rd.read(off, ln, files=files, stats=st)
    want = read_ref.read(buf, off, ln, files=files, stats=ost)
    assert goff.size == len(ranges) + 1 and int(goff[-1]) == got.size
    if files is not None:
        fo = np.concatenate([[0], np.cumsum(sizes)])
        off = off + fo[np.asarray(files)].astype(np.uint64)
    for r, (a, b) in enumerate(zip(off, ln)):
        g = got[int(goff[r]):int(goff[r + 1])].tobytes()
        assert g == data[int(a):int(a + b)].tobytes() == want[r], (kind, r, int(a), int(b))
    assert st == ost, (kind, st, ost)
    slots, recs = read_ref.touched(buf, off, ln)
    assert st["inflated"] == slots.size and st["deltas"] == recs.size
    return st


@pytest.mark.parametrize("kind", ["v1", "v2", "v3"])
def test_random_and_edge_ranges(ctx, archives, kind):
    data, ar, _, _ = archives[kind]
    raw = data.size
    rng = np.random.default_rng({"v1": 1, "v2": 2, "v3": 3}[kind])
    ends = _chunk_ends(ar)
    ranges = _edge_ranges(rng, ends, raw)
    ln = np.minimum((np.exp(rng.uniform(0, np.log(200 << 10), 300))).astype(np.int64), raw)
    ranges += [(int(rng.integers(0, raw - x + 1)), int(x)) for x in ln]
    ranges += [ranges[int(i)] for i in rng.integers(0, len(ranges), 40)]      # repeats
    ranges += [(a + b // 3, b // 2) for a, b in ranges[200:240]]              # overlaps
    order = rng.permutation(len(ranges))
    st = _check(ctx, kind, archives, [ranges[i] for i in order])
    assert st["inflated"] == ar.n_unique                                       # the whole stream is one of them
    # small batches inflate only what they touch
    k1, k2 = ends.size // 5, ends.size // 2
    few = [(int(ends[k1]) - 1, 2), (int(ends[k2]), 4096), (int(ends[k1]), 1)]
    st = _check(ctx, kind, archives, few)
    assert st["inflated"] <= 4


def test_deltas_and_their_bases_inflate_once(ctx, archives):
    data, ar, buf, _ = archives["v2"]
    pos = _positions(ar)
    ends = _chunk_ends(ar)
    starts = np.concatenate([[0], ends[:-1]])
    sb = ar.store.size
    dch = np.flatnonzero(pos >= sb)
    upos = np.concatenate([[0], np.cumsum(ar.index[:, 36:38].copy().view("<u2").reshape(-1).astype(np.int64))[:-1]])
    picked = []
    for c in dch[:: max(1, dch.size // 8)]:
        dp = int(pos[c]) - sb
        bslot = int(ar.delta_store[dp:dp + 4].copy().view("<u4")[0])
        direct = np.flatnonzero(pos == upos[bslot])
        picked.append((int(c), bslot, direct))
    ranges = []
    for c, bslot, direct in picked:
        cs, ce = int(starts[c]), int(ends[c])
        ranges.append((cs + 3, ce - cs - 6))                  # inside the delta chunk
        ranges.append((max(cs - 100, 0), min(ce + 100, data.size) - max(cs - 100, 0)))   # the delta chunk and its neighbours
        if direct.size:                                       # its base, read directly in the same batch
            b = int(direct[0])
            ranges.append((int(starts[b]), int(ends[b] - starts[b])))
            ranges.append((int(starts[b]) + 7, 1))
    assert any(d.size for _, _, d in picked)
    st = _check(ctx, "v2", archives, ranges)
    assert st["deltas"] >= len(picked)


def test_file_relative_ranges(ctx, archives):
    from hmse_b200 import archive
    data, ar, _, sizes = archives["v3"]
    rng = np.random.default_rng(4)
    f = rng.integers(0, sizes.size, 200)
    ln = (rng.random(200) * (sizes[f] + 1)).astype(np.int64)
    a = (rng.random(200) * (sizes[f] - ln + 1)).astype(np.int64)
    empty = np.flatnonzero(sizes == 0)
    f = np.concatenate([f, empty, [sizes.size - 2]])
    a = np.concatenate([a, np.zeros(empty.size, np.int64), [int(sizes[-2]) - 1]])
    ln = np.concatenate([ln, np.zeros(empty.size, np.int64), [1]])
    _check(ctx, "v3", archives, list(zip(a.tolist(), ln.tolist())), files=f)
    rd = archive.Reader(ar, ctx)
    with pytest.raises(IndexError):
        rd.read([0], [0], files=[sizes.size])
    with pytest.raises(IndexError):
        rd.read([0], [0], files=[-1])
    big = int(np.argmax(sizes))
    with pytest.raises(ValueError):
        rd.read([1], [int(sizes[big])], files=[big])
    with pytest.raises(ValueError):
        rd.read([0], [1], files=[int(empty[0])])
    with pytest.raises(ValueError):
        archive.Reader(archives["v1"][1], ctx).read([0], [1], files=[0])


def _raw_read(rd, ranges, out_cap, out=None):
    """hmse_read through ctypes: (rc, out, out_off, total, status, n_bad)."""
    import torch
    ctx = rd.ctx
    rr = ctx.stage_u64(np.asarray(ranges, dtype=np.uint64).reshape(-1))
    R = len(ranges)
    if out is None:
        out = torch.full((out_cap + 64,), 0xAA, dtype=torch.uint8, device=ctx.tdev)
    oo = torch.full((R + 1,), -1, dtype=torch.int64, device=ctx.tdev)
    status = torch.full((R,), 99, dtype=torch.int32, device=ctx.tdev)
    tot, bad = C.c_uint64(0), C.c_uint64(0)
    rc = ctx.lib.hmse_read(ctx.h, rd.layout.data_ptr(), rd.n, rd.m, rd.n_delta, rd.store.data_ptr(),
                           rd.dstore.data_ptr() if rd.n_delta else None, rd.zd.data_ptr() if rd.zd.numel() else None,
                           int(rd.zd.numel()), rr.data_ptr(), R, out.data_ptr(), out_cap, oo.data_ptr(), C.byref(tot),
                           status.data_ptr(), C.byref(bad), None, ctx.stream)
    return rc, out, oo, tot.value, status, bad.value


def test_damaged_stored_chunk_fails_only_its_ranges(ctx, archives):
    import copy
    from hmse_b200 import archive
    data, ar, buf, _ = archives["v1"]
    upos = np.concatenate([[0], np.cumsum(ar.index[:, 36:38].copy().view("<u2").reshape(-1).astype(np.int64))])
    s = ar.n_unique // 2
    bad = copy.copy(ar)
    bad.store = ar.store.copy()
    bad.store[int(upos[s] + upos[s + 1]) // 2] ^= 0x5A
    rd = archive.Reader(bad, ctx)                     # the records are intact
    pos, ends = _positions(ar), _chunk_ends(ar)
    starts = np.concatenate([[0], ends[:-1]])
    hit = np.flatnonzero(pos == upos[s])
    rng = np.random.default_rng(6)
    ranges = []
    for c in hit:
        ranges += [(int(starts[c]), int(ends[c] - starts[c])), (max(int(starts[c]) - 50, 0), 100), (int(ends[c]) - 1, 1)]
    ln = rng.integers(1, 30000, 200)
    ranges += [(int(rng.integers(0, data.size - x)), int(x)) for x in ln]
    ranges = [ranges[i] for i in rng.permutation(len(ranges))]
    total = sum(b for _, b in ranges)
    rc, out, oo, tot, status, nbad = _raw_read(rd, ranges, total)
    assert rc == 0 and tot == total
    status, oo, out = status.cpu().numpy(), oo.cpu().numpy(), out.cpu().numpy()
    need = np.array([np.isin(s, read_ref.touched(buf, [a], [b])[0]).item() for a, b in ranges])
    assert need.sum() >= 3 and (~need).sum() > 100
    assert np.array_equal(status != 0, need) and nbad == need.sum()
    assert set(status[need].tolist()) <= set(range(1, 7))
    for r, (a, b) in enumerate(ranges):
        if not need[r]:
            assert out[oo[r]:oo[r + 1]].tobytes() == data[a:a + b].tobytes()
    assert (out[total:] == 0xAA).all()                # nothing behind the packed output
    with pytest.raises(ValueError, match="damaged chunk"):
        rd.read([a for a, _ in ranges], [b for _, b in ranges])


def test_damaged_delta_gives_16_plus_its_code(ctx, archives):
    import copy
    from hmse_b200 import archive
    data, ar, buf, _ = archives["v2"]
    pos, ends = _positions(ar), _chunk_ends(ar)
    starts = np.concatenate([[0], ends[:-1]])
    sb = ar.store.size
    c = int(np.flatnonzero(pos >= sb)[3])
    dp = int(pos[c]) - sb
    bad = copy.copy(ar)
    bad.delta_store = ar.delta_store.copy()
    bad.delta_store[dp + 8] = 0xFF                     # an unterminated varint / op that runs past the delta
    bad.delta_store[dp + 9] = 0xFF
    rd = archive.Reader(bad, ctx)
    users = np.flatnonzero(pos == pos[c])                # the chunks stored as this record
    ranges = [(int(starts[u]), int(ends[u] - starts[u])) for u in users] + [(int(starts[users[0]]) + 1, 1)]
    rng = np.random.default_rng(8)
    ranges += [(int(x), 3000) for x in rng.integers(0, data.size - 3000, 300)]
    hits = lambda a, b: bool(((starts[users] < a + b) & (ends[users] > a)).any())   # noqa: E731
    total = sum(b for _, b in ranges)
    rc, out, oo, tot, status, nbad = _raw_read(rd, ranges, total)
    assert rc == 0
    status, oo, out = status.cpu().numpy(), oo.cpu().numpy(), out.cpu().numpy()
    for r, (a, b) in enumerate(ranges):
        if hits(a, b):
            assert 17 <= status[r] <= 21, (r, status[r])
        else:
            assert status[r] == 0 and out[oo[r]:oo[r + 1]].tobytes() == data[a:a + b].tobytes()
    assert nbad == int((status != 0).sum()) >= 1
    with pytest.raises(ValueError):
        archive.restore(bad, ctx=ctx)


def _open_fails(ctx, ar, what):
    from hmse_b200 import archive
    with pytest.raises(ValueError, match=what):
        archive.Reader(ar, ctx)
    with pytest.raises(ValueError):
        archive.restore(ar, ctx=ctx)


def test_damaged_records_fail_the_open(ctx, archives):
    import copy
    data, ar1, _, _ = archives["v1"]
    _, ar2, _, _ = archives["v2"]
    # (1) an index entry's lba off by one sector
    b = copy.copy(ar1)
    b.index = ar1.index.copy()
    b.index[5, 32:36] = (ar1.index[5, 32:36].copy().view("<u4") + 1).view(np.uint8)
    _open_fails(ctx, b, "tile")
    # (2) a pointer record's in-sector offset
    b = copy.copy(ar1)
    b.pointers = ar1.pointers.copy()
    b.pointers[7, 4] ^= 1
    _open_fails(ctx, b, "does not address a stored chunk")
    # (3) a DeltaChunk record whose base slot is >= m; a delta pointer in an archive without a delta store
    pos = _positions(ar2)
    dp = int(pos[np.flatnonzero(pos >= ar2.store.size)[0]]) - ar2.store.size
    b = copy.copy(ar2)
    b.delta_store = ar2.delta_store.copy()
    b.delta_store[dp:dp + 4] = np.array([ar2.n_unique], dtype="<u4").view(np.uint8)
    _open_fails(ctx, b, "DeltaChunk record is damaged")
    b = copy.copy(ar2)
    b.delta_store, b.n_delta = None, 0
    _open_fails(ctx, b, "delta store")
    # (4) two pointers to one stored chunk disagree on its length
    pos1 = _positions(ar1)
    u, cnt = np.unique(pos1, return_counts=True)
    dup = np.flatnonzero(pos1 == u[np.flatnonzero(cnt > 1)[0]])
    b = copy.copy(ar1)
    b.pointers = ar1.pointers.copy()
    raw = b.pointers[dup[1], 6:8].copy().view("<u2")
    b.pointers[dup[1], 6:8] = (raw - 1).view(np.uint8)
    _open_fails(ctx, b, "disagree")
    # (5) a stored chunk nobody references: one more index entry and its stream behind the store
    b = copy.copy(ar1)
    sb = ar1.store.size
    extra = ar1.index[0].copy()
    extra[32:36] = np.array([sb >> 9], dtype="<u4").view(np.uint8)
    b.index = np.concatenate([ar1.index, extra[None, :]])
    b.store = np.concatenate([ar1.store, ar1.store[:int(ar1.index[0, 36:38].copy().view("<u2")[0])]])
    b.pointers = ar1.pointers.copy()
    _open_fails(ctx, b, "no known raw length")
    # (6) the raw lengths do not add up to raw_bytes
    b = copy.copy(ar1)
    b.raw_bytes = ar1.raw_bytes + 1
    _open_fails(ctx, b, "add up")


def test_bad_ranges_and_capacity(ctx, archives):
    from hmse_b200 import archive, _lib
    data, ar, _, _ = archives["v1"]
    rd = archive.Reader(ar, ctx)
    raw = data.size
    for bad in ([(0, 10), (raw - 5, 6)], [(5, 10), (2 ** 64 - 1, 2)], [(raw + 1, 0)]):
        rc, out, oo, _, status, _ = _raw_read(rd, bad, 1 << 16)
        assert rc == _lib.HMSE_E_INVAL
        assert (out.cpu().numpy() == 0xAA).all() and (oo.cpu().numpy() == -1).all() and (status.cpu().numpy() == 99).all()
    with pytest.raises(ValueError):
        rd.read([raw - 5], [6])
    rc, out, oo, tot, status, _ = _raw_read(rd, [(0, 5000), (100, 20000)], 24999)
    assert rc == _lib.HMSE_E_CAPACITY and tot == 25000
    assert (out.cpu().numpy() == 0xAA).all() and (oo.cpu().numpy() == -1).all()
    rc, out, oo, tot, status, _ = _raw_read(rd, [(0, 5000), (100, 20000)], 25000)
    assert rc == 0 and out[:25000].cpu().numpy().tobytes() == data[:5000].tobytes() + data[100:20100].tobytes()
    # an empty batch, and a layout given the wrong archive size
    got, off = rd.read([], [])
    assert got.size == 0 and off.tolist() == [0]
    rr = ctx.stage_u64(np.array([0, 1], dtype=np.uint64))
    oo = ctx.empty(2, __import__("torch").int64)
    st = ctx.empty(1, __import__("torch").int32)
    tot = C.c_uint64(0)
    rc = ctx.lib.hmse_read(ctx.h, rd.layout.data_ptr(), rd.n - 1, rd.m, 0, rd.store.data_ptr(), None, rd.zd.data_ptr(),
                           int(rd.zd.numel()), rr.data_ptr(), 1, ctx.empty(64, __import__("torch").uint8).data_ptr(), 1,
                           oo.data_ptr(), C.byref(tot), st.data_ptr(), None, None, ctx.stream)
    assert rc == _lib.HMSE_E_INVAL


def test_launch_count_does_not_depend_on_the_batch(ctx, archives):
    from hmse_b200 import archive
    data, ar, _, _ = archives["v2"]
    rd = archive.Reader(ar, ctx)
    pos, ends = _positions(ar), _chunk_ends(ar)
    starts = np.concatenate([[0], ends[:-1]])
    c = int(np.flatnonzero(pos >= ar.store.size)[0])
    rng = np.random.default_rng(12)
    small = [(int(starts[c]), 100)] + [(int(rng.integers(0, data.size - 4096)), 4096) for _ in range(9)]
    ln = rng.integers(1, 8192, 100000)
    big = [(int(starts[c]), 100)] + [(int(rng.integers(0, data.size - x)), int(x)) for x in ln[1:]]
    counts = []
    for batch in (small, big, small):
        st = {}
        n0 = ctx.lib.hmse_launch_count(ctx.h)
        rd.read([a for a, _ in batch], [b for _, b in batch], stats=st)
        counts.append(ctx.lib.hmse_launch_count(ctx.h) - n0)
        assert st["inflated"] > 0 and st["deltas"] > 0
    assert counts[0] == counts[1] == counts[2], counts


@pytest.fixture(scope="module")
def big_archive(ctx):
    """256 MiB of the device corpus (seed 42) with repeats, ingested into an archive."""
    import torch
    import hmse_b200
    from hmse_b200 import archive
    from hmse_b200.corpus import DeviceCorpus
    zd = corpus.zdict()
    d = DeviceCorpus(ctx).generate(192 << 20)[:192 << 20]
    d = torch.cat([d, d[32 << 20:96 << 20]])
    ar = archive.build(hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(d)), zd, ctx=ctx)
    return d, ar


def test_a_million_ranges_in_one_call(ctx, big_archive):
    import torch
    from hmse_b200 import archive
    d, ar = big_archive
    raw = d.numel()
    rng = np.random.default_rng(1)
    R = 1_000_000
    ln = np.exp(rng.uniform(0, np.log(65536), R)).astype(np.int64)
    off = (rng.random(R) * (raw - ln + 1)).astype(np.int64)
    rd = archive.Reader(ar, ctx)
    st = {}
    got, goff = rd.read(off, ln, device_out=True, stats=st)
    assert goff.numel() == R + 1 and int(goff[-1]) == int(ln.sum()) == got.numel()
    # compare on the device in slices of ranges: output byte k of range r is input byte off[r] + k
    offd, lnd = torch.from_numpy(off).to(ctx.tdev), torch.from_numpy(ln).to(ctx.tdev)
    for a in range(0, R, 50000):
        b = min(a + 50000, R)
        l = lnd[a:b]
        base = torch.repeat_interleave(offd[a:b] - goff[a:b], l)
        idx = base + torch.arange(int(goff[a]), int(goff[b]), device=ctx.tdev)
        assert torch.equal(got[int(goff[a]):int(goff[b])], d[idx]), (a, b)
    slots, recs = read_ref.touched(ar.tobytes(), off, ln)
    assert st["inflated"] == slots.size and st["deltas"] == 0
    ulen = np.zeros(ar.n_unique, np.int64)
    upos = np.concatenate([[0], np.cumsum(ar.index[:, 36:38].copy().view("<u2").reshape(-1).astype(np.int64))[:-1]])
    pos = _positions(ar)
    raw_l = ar.pointers[:, 6:8].copy().view("<u2").reshape(-1).astype(np.int64) + 1
    ulen[np.searchsorted(upos, pos)] = raw_l
    assert st["inflated_bytes"] == int(ulen[slots].sum())


def test_scratch_follows_the_batch(ctx, big_archive):
    import hmse_b200
    from hmse_b200 import archive
    _, ar = big_archive
    fresh = hmse_b200.Context(0)
    rd = archive.Reader(ar, fresh)
    s0 = fresh.lib.hmse_scratch_bytes(fresh.h)
    rng = np.random.default_rng(3)
    got, _ = rd.read(rng.integers(0, ar.raw_bytes - 4096, 10), np.full(10, 4096))
    grow = fresh.lib.hmse_scratch_bytes(fresh.h) - s0
    assert got.size == 40960
    assert grow < ar.store.size // 20, (grow, ar.store.size)
    fresh.close()


def test_reads_past_2_32(ctx):
    """A 4.5 GB stream of tiled corpus (the store stays small): ranges below, across and above 2^32, and an output
    larger than 2^32 bytes."""
    import torch
    import hmse_b200
    from hmse_b200 import archive
    from hmse_b200.corpus import DeviceCorpus
    zd = corpus.zdict()
    tile = DeviceCorpus(ctx).generate(48 << 20)[:48 << 20]
    d = tile.repeat(96)                                       # 4.5 GiB
    d = torch.cat([d, tile[:12345]])
    ar = archive.build(hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(d)), zd, ctx=ctx)
    assert ar.raw_bytes == d.numel() > (1 << 32) + (256 << 20)
    rd = archive.Reader(ar, ctx)
    T = 1 << 32
    ranges = [(T - 4096, 4096), (T - 1, 2), (T, 1), (T - 100000, 300000), (T + 12345, 65536), (ar.raw_bytes - 7, 7),
              (T - 1, 1), (2 << 30, (2 << 30) + 4096), (1000, T + 5000)]
    got, off = rd.read([a for a, _ in ranges], [b for _, b in ranges], device_out=True)
    for r, (a, b) in enumerate(ranges):
        assert torch.equal(got[int(off[r]):int(off[r + 1])], d[a:a + b]), r
    whole = archive.restore(ar, ctx=ctx, device_out=True)
    assert whole.numel() == d.numel() and torch.equal(whole, d)
