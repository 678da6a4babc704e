"""GPU: many files in one call (hmse_chunk_files) - every file is chunked exactly as hmse_chunk chunks it alone
(tests/files_ref.py runs the oracle on each file's bytes by themselves), through ingest, dedup, L4 and the v3 archive
with its per-file restore."""
import ctypes as C

import numpy as np
import pytest

import oracle
from oracle import corpus
from oracle.config import CDCConfig as OCfg
from tests import files_ref

pytestmark = pytest.mark.gpu

TINY = OCfg(64, 256, 1024, oracle.config.spread_mask(10), oracle.config.spread_mask(6))


def _pcfg(o: OCfg):
    import hmse_b200
    return hmse_b200.CDCConfig(o.min_size, o.avg_size, o.max_size, o.mask_s, o.mask_l, o.gear_seed)


def _seg_len(o: OCfg):
    return max(8 * o.max_size, 256 << 10)


def _compare(got, want, what, off=None):
    if np.array_equal(got, want):
        return
    k = min(got.size, want.size)
    bad = np.flatnonzero(got[:k] != want[:k])
    first = int(bad[0]) if bad.size else k
    where = ""
    if off is not None and first < want.size:
        f = int(np.searchsorted(off, int(want[first]), side="left")) - 1
        where = " (file %d = [%d, %d))" % (f, int(off[f]), int(off[f + 1]))
    raise AssertionError("%s differ: got %d want %d first mismatch @%d%s got %s want %s" % (
        what, got.size, want.size, first, where, got[max(0, first - 1):first + 3], want[max(0, first - 1):first + 3]))


def _check(ctx, data, sizes, ocfg=OCfg()):
    import hmse_b200
    data = np.ascontiguousarray(data, dtype=np.uint8)
    sizes = np.asarray(sizes, dtype=np.int64)
    got, gfc = hmse_b200.chunk_files(data, sizes, _pcfg(ocfg), ctx=ctx)
    want, wfc = files_ref.chunk_files(data, sizes, ocfg)
    assert got.dtype == np.uint64 and gfc.dtype == np.uint64
    off = np.concatenate([[0], np.cumsum(sizes)])
    _compare(got, want, "cuts", off)
    _compare(gfc, wfc, "file_chunk")
    return got, gfc


def _log_uniform(rng, n_files, hi):
    s = (np.exp(rng.uniform(0, np.log(hi + 1), n_files)) - 1).astype(np.int64)
    r = rng.random(n_files)
    s[r < 0.2] = 0
    s[(r >= 0.2) & (r < 0.3)] = 1
    return s


def _fit(sizes, n):
    """The prefix of `sizes` that fits in n bytes, with the last file cut to fill them exactly."""
    c = np.cumsum(sizes)
    assert c[-1] >= n
    k = int(np.searchsorted(c, n))
    out = sizes[:k + 1].copy()
    out[-1] = n - (int(c[k - 1]) if k else 0)
    return out


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_mixes_over_corpus(ctx, corpus8, seed):
    rng = np.random.default_rng(seed)
    data = np.tile(corpus8, 4)
    sizes = _fit(_log_uniform(rng, 4000, 1 << 20), data.size)
    assert (sizes == 0).sum() > 20 and (sizes == 1).sum() > 10
    _check(ctx, data, sizes)


def test_boundary_sizes(ctx, corpus8):
    o = OCfg()
    sl = _seg_len(o)
    edge = [o.min_size - 1, o.min_size, o.min_size + 1, o.avg_size, o.max_size - 1, o.max_size, o.max_size + 1,
            sl - 1, sl, sl + 1, 0, 1, 2 * sl + 1]
    sizes = np.array(edge * 3, dtype=np.int64)
    _check(ctx, corpus8[:int(sizes.sum())], sizes)


def test_one_file_spanning_many_segments(ctx, corpus8):
    n = corpus8.size
    sizes = np.array([1000, n - 3000, 0, 2000], dtype=np.int64)
    _check(ctx, corpus8, sizes)


@pytest.mark.parametrize("ocfg", [OCfg.for_avg(4096), TINY], ids=["spec_1_4_16", "tiny_64_256_1024"])
def test_other_configs(ctx, corpus8, ocfg):
    rng = np.random.default_rng(11)
    sizes = _fit(_log_uniform(rng, 3000, 256 << 10), 4 << 20)
    sizes = np.concatenate([sizes[:-1], [ocfg.min_size - 1, ocfg.min_size, ocfg.min_size + 1, ocfg.max_size + 1, _seg_len(ocfg) + 1],
                            [sizes[-1]]])
    _check(ctx, corpus8[:int(sizes.sum())], sizes, ocfg)


def test_random_bytes(ctx):
    d = corpus.random_bytes(4 << 20)
    sizes = _fit(_log_uniform(np.random.default_rng(5), 3000, 1 << 20), d.size)
    _check(ctx, d, sizes)


def test_zero_runs(ctx, corpus8):
    # a file of zeros, and a zero run that straddles a file boundary: max-size cuts at phases no guess knows
    d = corpus8[:6 << 20].copy()
    d[(1 << 20) + 777:(4 << 20) + 123] = 0
    sizes = np.array([(2 << 20) + 5, (3 << 20) - 11, 1, 0, d.size - (5 << 20) - 1 + 6], dtype=np.int64)
    sizes[-1] = d.size - int(sizes[:-1].sum())
    _check(ctx, d, sizes)
    _check(ctx, np.zeros(3 << 20, np.uint8), [1 << 20, 12345, (2 << 20) - 12345])


def test_hundred_thousand_small_files(ctx, corpus8):
    rng = np.random.default_rng(9)
    sizes = rng.integers(64, 8193, 100_000)
    n = int(sizes.sum())
    data = np.tile(corpus8, n // corpus8.size + 1)[:n]
    _check(ctx, data, sizes)


def test_one_file_equals_chunk(ctx, corpus8):
    import torch
    import hmse_b200
    cfg = hmse_b200.CDCConfig()
    for n in (0, 1, 2047, 2049, 100000, corpus8.size):
        d = ctx.stage(corpus8[:n])
        want = ctx.chunk(d, cfg).clone()
        got, fc = ctx.chunk_files(d, torch.tensor([0, n], dtype=torch.int64, device=ctx.tdev), cfg)
        assert torch.equal(got, want), n
        assert fc.tolist() == [0, want.numel()]


def test_file_chunk_of_empty_files(ctx, corpus8):
    import torch
    import hmse_b200
    sizes = [0, 0, 5000, 0, 1, 0, 0, 70000, 0]
    d = corpus8[:sum(sizes)]
    cuts, fc = _check(ctx, d, sizes)
    f = fc.tolist()
    assert f[0] == f[1] == f[2] == 0 and f[3] == f[4] and f[5] == f[6] == f[7] and f[8] == f[9] == cuts.size   # empty files
    assert 0 < f[4] < f[7] < f[8]
    # device in, device out; empty input
    dc, dfc = hmse_b200.chunk_files(ctx.stage(d), torch.tensor(sizes, device=ctx.tdev), ctx=ctx)
    assert dc.is_cuda and np.array_equal(dc.cpu().numpy().view(np.uint64), cuts) and dfc.tolist() == fc.tolist()
    c0, f0 = hmse_b200.chunk_files(np.zeros(0, np.uint8), [0, 0], ctx=ctx)
    assert c0.size == 0 and f0.tolist() == [0, 0, 0]
    c0, f0 = hmse_b200.chunk_files(np.zeros(0, np.uint8), [], ctx=ctx)
    assert c0.size == 0 and f0.tolist() == [0]


def test_offsets_past_4_gib(ctx):
    """A 4.5 GB buffer of device-rendered corpus split into files: the files around 2^32 (one of them straddles it) equal
    the oracle run on their own bytes."""
    import torch
    import hmse_b200
    from hmse_b200 import corpus as pc
    n = 4_500_000_000
    rng = np.random.default_rng(4)
    t = 1 << 32
    head = _fit(_log_uniform(rng, 100000, 1 << 20), t - (40 << 20))
    around = np.array([1, 0, 3 << 20, 77777, 64 << 20, 0, 5, 2048, 1 << 20], dtype=np.int64)   # the 64 MiB file straddles 2^32
    tail = _fit(_log_uniform(rng, 100000, 1 << 20), n - int(head.sum()) - int(around.sum()))
    sizes = np.concatenate([head, around, tail])
    assert int(sizes.sum()) == n
    off = np.concatenate([[0], np.cumsum(sizes)])
    d = pc.DeviceCorpus(ctx).generate(n)
    cfg = hmse_b200.CDCConfig()
    cuts, fc = ctx.chunk_files(d, torch.from_numpy(off).to(ctx.tdev), cfg)
    cuts = cuts.cpu().numpy().view(np.uint64)
    fc = fc.cpu().numpy()
    assert fc[-1] == cuts.size and int(cuts[-1]) == n
    f0 = head.size - 2
    f1 = head.size + around.size + 2
    assert off[f0] < t - (8 << 20) and off[f1] > t + (8 << 20)
    straddle = int(np.searchsorted(off, t, side="right")) - 1
    assert off[straddle] < t < off[straddle + 1] and sizes[straddle] == 64 << 20
    host = d[int(off[f0]):int(off[f1])].cpu().numpy()
    for f in range(f0, f1):
        want = oracle.chunk_c(host[off[f] - off[f0]:off[f + 1] - off[f0]]) + np.uint64(off[f])
        _compare(cuts[fc[f]:fc[f + 1]], want, "cuts of file %d" % f)
    del d
    torch.cuda.empty_cache()


def test_scratch_is_linear_in_bytes_and_files(ctx):
    """Scratch after chunk_files of 10^6 small files: the bitmaps (a quarter of the bytes), the cut lists (8 bytes per
    min_size bytes + 16 per segment) and about 120 bytes of records per file - not a cut list of seg_len / min_size
    entries per file."""
    import torch
    import hmse_b200
    c = hmse_b200.Context(0)
    try:
        rng = np.random.default_rng(3)
        sizes = rng.integers(1, 300, 1_000_000)
        n = int(sizes.sum())
        d = hmse_b200.corpus.DeviceCorpus(c).generate(n)
        cfg = hmse_b200.CDCConfig()
        before = c.lib.hmse_scratch_bytes(c.h)
        cuts, fc = c.chunk_files(d, torch.from_numpy(np.concatenate([[0], np.cumsum(sizes)])).to(c.tdev), cfg)
        assert cuts.numel() == 1_000_000 and int(fc[-1]) == 1_000_000
        grown = c.lib.hmse_scratch_bytes(c.h) - before
        bound = 1.25 * (n / 4 + 8 * n / cfg.min_size + 160 * sizes.size) + (8 << 20)
        assert grown <= bound, "scratch grew by %d bytes, bound %d" % (grown, bound)
    finally:
        c.close()


def test_context_state_after_chunk_files(ctx, corpus8):
    """chunk_files, then the virtual-shard sequence of test_gpu_cdc.py (speculative resolve, then the true entry): the
    incremental re-resolve must not reuse segment records of the file table."""
    import hmse_b200
    cfg = hmse_b200.CDCConfig()
    d = corpus8[:6 << 20]
    n = d.size
    want = oracle.chunk_c(d)
    dev = ctx.stage(d)
    for world in (2, 3):
        sizes = _fit(_log_uniform(np.random.default_rng(world), 3000, 64 << 10), n)
        _check(ctx, d, sizes)
        per = (n + world - 1) // world
        got, entry = [], 0
        for r in range(world):
            lo, hi = r * per, min(n, (r + 1) * per)
            eof = hi == n
            avail_hi = n if eof else min(n, hi + cfg.max_size)
            if not eof and avail_hi - lo < (hi - lo) + cfg.max_size:
                eof = True
                avail_hi = n
            buf = ctx.stage(dev[lo:avail_hi].clone())
            ctx.chunk_scan(buf, cfg)
            ctx.chunk_resolve(buf, cfg, hi - lo, eof, 0)
            # a file table in between: the next resolve must not take its records for this shard's
            ctx.chunk_files(ctx.stage(d[:1 << 20]), ctx.stage_u64([0, 1000, 1 << 20]), cfg)
            ctx.chunk_scan(buf, cfg)
            ctx.chunk_resolve(buf, cfg, hi - lo, eof, 0)
            cuts, ex = ctx.chunk_resolve(buf, cfg, hi - lo, eof, entry)
            got.append(cuts.cpu().numpy().view(np.uint64) + np.uint64(lo))
            if eof:
                break
            entry = ex - (hi - lo)
        assert np.array_equal(np.concatenate(got), want)


def test_bad_offsets_are_rejected(ctx, corpus8):
    import torch
    import hmse_b200
    cfg = hmse_b200.CDCConfig()
    d = ctx.stage(corpus8[:1 << 20])
    n = d.numel()
    cuts = ctx.empty(n // cfg.min_size + 10, torch.int64)
    fc = ctx.empty(8, torch.int64)
    for off in ([5, 1000, n], [0, 5000, 4000, n], [0, 1000, n + 1], [0, 1000, n - 1], [0, 1 << 62, n], [1]):
        o = ctx.stage_u64(off)
        nc = C.c_uint64(0)
        cuts.fill_(-7)
        rc = ctx.lib.hmse_chunk_files(ctx.h, d.data_ptr(), n, o.data_ptr(), len(off) - 1, C.byref(ctx.cdc_struct(cfg)),
                                      cuts.data_ptr(), cuts.numel(), C.byref(nc), fc.data_ptr(), ctx.stream)
        assert rc == hmse_b200._lib.HMSE_E_INVAL, (off, rc)
        assert "offsets" in ctx.lib.hmse_last_error(ctx.h).decode()
        assert bool((cuts == -7).all())
    torch.cuda.synchronize()
    _check(ctx, corpus8[:1 << 20], [1000, 0, (1 << 20) - 1000])
    # too small a capacity reports what is needed
    nc = C.c_uint64(0)
    o = ctx.stage_u64([0, n])
    rc = ctx.lib.hmse_chunk_files(ctx.h, d.data_ptr(), n, o.data_ptr(), 1, C.byref(ctx.cdc_struct(cfg)), cuts.data_ptr(), 3,
                                  C.byref(nc), fc.data_ptr(), ctx.stream)
    assert rc == hmse_b200._lib.HMSE_E_CAPACITY and nc.value == oracle.chunk_c(corpus8[:1 << 20]).size


def _files_dataset(seed=21):
    """corpus files plus 20 exact copies of earlier files, shuffled in."""
    rng = np.random.default_rng(seed)
    base = corpus.generate(3 << 20)
    sizes = _fit(_log_uniform(rng, 400, 256 << 10), base.size)
    off = np.concatenate([[0], np.cumsum(sizes)])
    files = [base[off[f]:off[f + 1]] for f in range(sizes.size)]
    for f in rng.choice(sizes.size, 20, replace=False):
        files.insert(int(rng.integers(0, len(files))), files[int(f)])
    return np.concatenate(files), np.array([x.size for x in files], dtype=np.int64)


def test_ingest_with_files_equals_oracle(ctx):
    import hmse_b200
    zd = corpus.zdict()
    data, sizes = _files_dataset()
    r = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(data), files=sizes)
    want, wfc = files_ref.chunk_files(data, sizes)
    _compare(r.cuts.cpu().numpy().view(np.uint64), want, "cuts")
    _compare(r.file_chunk.cpu().numpy().view(np.uint64), wfc, "file_chunk")
    wd = oracle.digest(data, want)
    assert np.array_equal(r.digests.cpu().numpy(), wd)
    wc, wf = oracle.dedup(wd)
    assert np.array_equal(r.canon.cpu().numpy(), wc) and np.array_equal(r.is_first.cpu().numpy(), wf)
    # without files nothing changes
    r0 = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(data))
    assert r0.file_chunk is None and np.array_equal(r0.cuts.cpu().numpy().view(np.uint64), oracle.chunk_c(data))


def test_small_duplicate_files_are_stored_once(ctx):
    import hmse_b200
    rng = np.random.default_rng(77)
    cfg = hmse_b200.CDCConfig()
    files = [corpus.random_bytes(int(rng.integers(1, cfg.min_size)), seed=1000 + i) for i in range(1000)]
    order = rng.permutation(2000)
    seq = [files[i % 1000] for i in order]
    data = np.concatenate(seq)
    sizes = np.array([x.size for x in seq], dtype=np.int64)
    r = hmse_b200.Ingest(ctx, cfg, b"").run(ctx.stage(data), files=sizes, compress=False)
    assert r.n_chunks == 2000 and r.file_chunk.tolist() == list(range(2001))
    first = r.is_first.cpu().numpy()
    canon = r.canon.cpu().numpy()
    assert first.sum() == 1000
    seen = {}
    for k, i in enumerate(order):
        f = int(i % 1000)
        if f in seen:
            assert not first[k] and canon[k] == seen[f]
        else:
            assert first[k]
            seen[f] = k
    # the same bytes as one stream: chunks span files, and the copies are not found
    r1 = hmse_b200.Ingest(ctx, cfg, b"").run(ctx.stage(data), compress=False)
    assert int(r1.is_first.sum()) > r1.n_chunks - 100 and r1.n_chunks < 1000


def test_ingest_files_with_l4_equals_oracle(ctx):
    import hmse_b200
    rng = np.random.default_rng(8)
    base = corpus.generate(2 << 20)
    near = base[:1 << 20].copy()
    near[500::40000] ^= 0x20
    data = np.concatenate([base, near, corpus.random_bytes(3000, seed=3)])
    sizes = np.concatenate([[1, 2, 3, 0, 3], _fit(_log_uniform(rng, 2000, 128 << 10), data.size - 9)])
    r = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), corpus.zdict()).run(ctx.stage(data), l4=hmse_b200.SimConfig(), files=sizes)
    cuts, _ = files_ref.chunk_files(data, sizes)
    lens = np.diff(np.concatenate([[0], cuts.astype(np.int64)]))
    assert (lens < 4).sum() >= 3                      # chunks without a shingle
    _compare(r.cuts.cpu().numpy().view(np.uint64), cuts, "cuts")
    _, first = oracle.dedup(oracle.digest(data, cuts))
    keys = oracle.band_keys(oracle.minhash_c(data, cuts))
    wbase, wblob, woffs = oracle.delta(data, cuts, keys, first)
    assert (wbase >= 0).sum() > 3
    assert np.array_equal(r.base.cpu().numpy(), wbase) and np.array_equal(r.delta_blob.cpu().numpy(), wblob)
    assert np.array_equal(r.delta_offsets.cpu().numpy().view(np.uint64), woffs)


@pytest.mark.parametrize("l4", [False, True])
def test_archive_v3_and_per_file_restore(ctx, l4):
    import struct
    import hmse_b200
    from hmse_b200 import archive
    zd = corpus.zdict()
    data, sizes = _files_dataset(seed=31)
    if l4:
        near = data[:1 << 20].copy()
        near[300::30000] ^= 0x20
        data, sizes = np.concatenate([data, near]), np.concatenate([sizes, [near.size]])
    sizes = np.concatenate([[0], sizes, [0]])
    off = np.concatenate([[0], np.cumsum(sizes)])
    ing = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd)
    r = ing.run(ctx.stage(data), files=sizes, l4=hmse_b200.SimConfig() if l4 else None)
    if l4:
        assert int((r.base >= 0).sum()) > 0
    ar = archive.build(r, zd, ctx=ctx)
    buf = ar.tobytes()
    assert struct.unpack_from("<I", buf, 8)[0] == 3 and ar.n_files == sizes.size
    back = archive.Archive.frombytes(buf)
    assert np.array_equal(back.file_chunk, r.file_chunk.cpu().numpy().astype(np.uint64))
    assert archive.restore(back, ctx=ctx).tobytes() == data.tobytes()
    assert files_ref.restore(buf) == data.tobytes()
    fc = back.file_chunk.astype(np.int64)
    ptr = back.pointers
    pos = ptr[:, 0:4].copy().view("<u4").reshape(-1).astype(np.int64) * 512 + ptr[:, 4:6].copy().view("<u2").reshape(-1)
    rng = np.random.default_rng(5)
    picks = [[0], [sizes.size - 1], list(rng.choice(sizes.size, 7, replace=False)), [int(np.argmax(sizes))], [3, 3]]
    if l4:
        dchunks = np.flatnonzero(pos >= back.store.size)
        picks.append([int(np.searchsorted(fc, dchunks[0], side="right")) - 1])
    for sel in picks:
        st, ost = {}, {}
        got = archive.restore(back, ctx=ctx, files=sel, stats=st)
        assert [g.tobytes() for g in got] == [data[off[f]:off[f + 1]].tobytes() for f in sel]
        assert files_ref.restore(buf, files=sel, stats=ost) == [g.tobytes() for g in got]
        rows = np.concatenate([np.arange(fc[f], fc[f + 1]) for f in sel]) if sel else np.zeros(0, np.int64)
        # no more streams than the files reference: their stored chunks (and delta bases)
        n_ref = np.unique(pos[rows]).size
        assert st["inflated"] <= n_ref + st["deltas"], (sel, st, n_ref)
        assert st["inflated"] == ost["inflated"], (sel, st, ost)
        assert st["inflated"] < back.n_unique
    # damaged file tables are rejected
    t = len(buf) - 8 * fc.size
    for k, v in ((0, 1), (2, int(fc[1]) + 10**6), (fc.size - 1, int(fc[-1]) - 1), (-1, fc.size)):
        bad = bytearray(buf)
        struct.pack_into("<Q", bad, t + 8 * k, v)
        with pytest.raises(ValueError):
            archive.Archive.frombytes(bytes(bad))
    for bad in (buf[:-8], buf + b"\0" * 8):
        with pytest.raises(ValueError):
            archive.Archive.frombytes(bad)
    # the same inputs without files: v1 / v2, unchanged, and no file table to restore from
    r0 = ing.run(ctx.stage(data), l4=hmse_b200.SimConfig() if l4 else None)
    a0 = archive.build(r0, zd, ctx=ctx)
    b0 = a0.tobytes()
    cuts0 = r0.cuts.cpu().numpy().view(np.uint64)
    if l4:
        idx, p0, dstore, nd = oracle.archive.records_l4(r0.digests.cpu().numpy(), r0.canon.cpu().numpy(), cuts0,
                                                        r0.select.cpu().numpy(), r0.offsets.cpu().numpy().view(np.uint64),
                                                        r0.base.cpu().numpy(), r0.delta_blob.cpu().numpy(),
                                                        r0.delta_offsets.cpu().numpy().view(np.uint64))
        assert b0 == oracle.archive.pack(zd, idx, p0, r0.blob.cpu().numpy(), data.size, dstore, nd)
        assert struct.unpack_from("<I", b0, 8)[0] == 2
    else:
        idx, p0 = oracle.archive.records(r0.digests.cpu().numpy(), r0.canon.cpu().numpy(), cuts0, r0.select.cpu().numpy(),
                                         r0.offsets.cpu().numpy().view(np.uint64))
        assert b0 == oracle.archive.pack(zd, idx, p0, r0.blob.cpu().numpy(), data.size)
        assert struct.unpack_from("<I", b0, 8)[0] == 1
    assert archive.Archive.frombytes(b0).file_chunk is None
    with pytest.raises(ValueError):
        archive.restore(a0, ctx=ctx, files=[0])
