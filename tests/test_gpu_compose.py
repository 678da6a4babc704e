"""Composing archives on the device (hmse_compose, archive.compose): merges and subsets of archives ingested separately are
byte for byte the archive of one ingest of the selected files; with deltas the output equals the CPU reference
(tests/compose_ref.py), opens, and restores every selected file; dedup works across archives and refcounts saturate;
stores past 2^32 bytes; bad input is rejected before anything is written; the kernel count does not depend on the
number of sources or runs."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from oracle import corpus
from tests import compose_ref

pytestmark = pytest.mark.gpu


def _ingest(ctx, files, l4=False):
    import hmse_b200
    from hmse_b200 import archive
    zd = corpus.zdict()
    data = np.concatenate(files)
    res = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(data), files=[f.size for f in files],
                                                                l4=hmse_b200.SimConfig() if l4 else None)
    return archive.build(res, zd, ctx=ctx)


def _mix(corpus8, seed, n):
    """n files cut from random places of the corpus (overlaps, so chunks repeat across files), some empty, some copies."""
    rng = np.random.default_rng(seed)
    files = []
    for k in range(n):
        size = int(rng.integers(0, 96 << 10)) if rng.random() > 0.1 else 0
        a = int(rng.integers(0, corpus8.size - size))
        files.append(corpus8[a:a + size] if rng.random() > 0.1 or not files else files[int(rng.integers(0, len(files)))])
    return files


@pytest.mark.parametrize("groups", [2, 3])
def test_merge_equals_one_ingest(ctx, corpus8, groups):
    from hmse_b200 import archive
    files = _mix(corpus8, groups, 90)
    files[0] = corpus8[:40000]
    files[-3:] = files[:3]   # copies in the first and the last archive: chunks shared across archives
    bounds = [0, *np.sort(np.random.default_rng(groups).choice(np.arange(1, 90), groups - 1, replace=False)).tolist(), 90]
    srcs = [_ingest(ctx, files[a:b]) for a, b in zip(bounds[:-1], bounds[1:])]
    st = {}
    got = archive.compose([(s, None) for s in srcs], ctx=ctx, stats=st)
    want = _ingest(ctx, files)
    assert got.tobytes() == want.tobytes()
    assert st["stored"] == want.n_unique and st["deduplicated"] == st["stored_referenced"] - want.n_unique > 0


def test_subset_with_reorder_and_repeats(ctx, corpus8):
    from hmse_b200 import archive
    files = _mix(corpus8, 7, 80)
    a, b = _ingest(ctx, files[:40]), _ingest(ctx, files[40:])
    rd = archive.Reader(b, ctx)
    rng = np.random.default_rng(1)
    s1, s2, s3 = rng.integers(0, 40, 25).tolist() + [3, 3], rng.integers(0, 40, 20).tolist(), [9, 0, 9]
    got = archive.compose([(a, s1), (rd, s2), (a, s3)], ctx=ctx)
    want = _ingest(ctx, [files[f] for f in s1] + [files[40 + f] for f in s2] + [files[f] for f in s3])
    assert got.tobytes() == want.tobytes()


def test_v1_source_is_one_file(ctx, corpus8):
    import hmse_b200
    from hmse_b200 import archive
    zd = corpus.zdict()
    whole = corpus8[1 << 20:3 << 20]
    v1 = archive.build(hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(whole)), zd, ctx=ctx)
    assert v1.file_chunk is None
    files = _mix(corpus8, 3, 30)
    b = _ingest(ctx, files)
    got = archive.compose([(b, [4, 2]), (v1, None), (b, None)], ctx=ctx)
    assert got.tobytes() == _ingest(ctx, [files[4], files[2], whole] + files).tobytes()


@pytest.fixture(scope="module")
def l4_sources(ctx, corpus8):
    import hmse_b200
    from hmse_b200 import archive
    zd = corpus.zdict()
    d2 = np.concatenate([corpus8[:6 << 20], corpus8[2 << 20:3 << 20]])
    v2 = archive.build(hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(d2), l4=hmse_b200.SimConfig()), zd, ctx=ctx)
    assert v2.n_delta > 20 and v2.file_chunk is None
    rng = np.random.default_rng(4)
    sizes = rng.integers(0, 256 << 10, 40)
    sizes[rng.random(40) < 0.15] = 0
    sizes[-1] = 0
    sizes[-1] = d2.size - int(sizes.sum())
    assert sizes[-1] > 0
    off = np.concatenate([[0], np.cumsum(sizes)])
    files = [d2[off[f]:off[f + 1]] for f in range(40)]
    v3 = _ingest(ctx, files, l4=True)
    assert v3.n_delta > 20
    return d2, v2, files, v3


def test_l4_sources(ctx, l4_sources):
    from hmse_b200 import archive
    d2, v2, files, v3 = l4_sources
    sel = [39, 5, 5, 17, 0, 28, 33, 12]
    parts = [(v3, sel), (v2, None), (v3, None)]
    st = {}
    got = archive.compose(parts, ctx=ctx, stats=st)
    assert got.tobytes() == compose_ref.compose([(s.tobytes(), f) for s, f in parts])
    assert st["records"] == got.n_delta > 0
    archive.Reader(got, ctx)   # every open check passes
    want = [files[f] for f in sel] + [d2] + files
    out = archive.restore(got, ctx=ctx, files=list(range(len(want))))
    assert all(np.array_equal(o, w) for o, w in zip(out, want))
    assert archive.compose([(v3, None)], ctx=ctx).tobytes() == v3.tobytes()


def test_cross_archive_dedup(ctx, corpus8):
    from hmse_b200 import archive
    files = _mix(corpus8, 21, 50)
    a = _ingest(ctx, files)
    st = {}
    got = archive.compose([(a, None), (a, None)], ctx=ctx, stats=st)
    assert np.array_equal(got.store, a.store) and np.array_equal(got.index[:, :32], a.index[:, :32])
    twice = _ingest(ctx, files + files)
    assert got.tobytes() == twice.tobytes()
    assert st["deduplicated"] == a.n_unique and st["stored"] == a.n_unique


def test_refcount_saturates(ctx, corpus8):
    from hmse_b200 import archive
    small = corpus8[5000:8000]
    a = _ingest(ctx, [small, corpus8[:50000]])
    assert int(a.file_chunk[1]) == 1
    got = archive.compose([(a, [0] * 70000)], ctx=ctx)
    assert got.n_unique == 1 and got.n_chunks == 70000
    assert int(got.index[0, 38:40].view("<u2")[0]) == 65535
    assert got.tobytes() == _ingest(ctx, [small] * 70000).tobytes()


def test_store_past_2_32(ctx):
    import torch
    import hmse_b200
    from hmse_b200 import archive
    zd = corpus.zdict()
    g = torch.Generator(device=ctx.tdev).manual_seed(5)
    n = 2_200_000_000
    srcs, datas = [], []
    for _ in range(2):
        d = torch.randint(0, 256, (n,), dtype=torch.uint8, device=ctx.tdev, generator=g)
        res = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(d), files=[n])
        srcs.append(archive.build(res, zd, ctx=ctx))
        datas.append(d.cpu())
        del res, d
    got = archive.compose([(srcs[0], None), (srcs[1], None)], ctx=ctx)
    assert got.store.size > (1 << 32) and got.raw_bytes == 2 * n
    pos = got.pointers[:, 0:4].copy().view("<u4").reshape(-1).astype(np.int64) * 512 + got.pointers[:, 4:6].copy().view("<u2").reshape(-1)
    c = int(np.searchsorted(pos, 1 << 32))
    raw_off = np.concatenate([[0], np.cumsum(got.pointers[:, 6:8].copy().view("<u2").reshape(-1).astype(np.int64) + 1)])
    x = int(raw_off[c])
    ranges = [(x - 100000, 300000), (x - 1, 2), (n - 5000, 10000), (2 * n - 4096, 4096)]
    rd = archive.Reader(got, ctx)
    out, off = rd.read([a for a, _ in ranges], [b for _, b in ranges])
    whole = torch.cat(datas).numpy()
    for r, (a, b) in enumerate(ranges):
        assert np.array_equal(out[int(off[r]):int(off[r + 1])], whole[a:a + b]), r


def test_errors(ctx, corpus8):
    import hmse_b200
    from hmse_b200 import archive
    zd = corpus.zdict()
    a = _ingest(ctx, [corpus8[:8 << 20], corpus8[:1000]])
    v1 = archive.build(hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(corpus8[:1 << 20])), zd, ctx=ctx)
    with pytest.raises(ValueError):
        archive.compose([(a, None), (dataclasses.replace(a, zdict=zd[:-1]), None)], ctx=ctx)
    with pytest.raises(IndexError):
        archive.compose([(a, [0, 2])], ctx=ctx)
    with pytest.raises(IndexError):
        archive.compose([(a, [-1])], ctx=ctx)
    with pytest.raises(ValueError):
        archive.compose([(v1, [0])], ctx=ctx)
    c = int(a.file_chunk[1])
    n0 = ctx.lib.hmse_launch_count(ctx.h)
    with pytest.raises(ValueError, match="2\\^32"):
        archive.compose([(a, [0] * ((0xFFFFFFFE // c) + 1))], ctx=ctx)
    assert ctx.lib.hmse_launch_count(ctx.h) == n0


def _desc(rds):
    from hmse_b200 import _lib
    descs = (_lib.ComposeSrc * len(rds))()
    for d, rd in zip(descs, rds):
        d.d_layout, d.d_index, d.d_pointers = rd.layout.data_ptr(), rd.index.data_ptr(), rd.pointers.data_ptr()
        d.d_store, d.d_delta_store = rd.store.data_ptr(), rd.dstore.data_ptr() if rd.n_delta else None
        d.n, d.m, d.n_delta = rd.n, rd.m, rd.n_delta
    return descs


def test_c_abi_capacity_and_bad_runs(ctx, l4_sources):
    import torch
    from hmse_b200 import _lib, archive
    _, v2, _, v3 = l4_sources
    rds = [archive.Reader(v2, ctx), archive.Reader(v3, ctx)]
    st = {}
    want = archive.compose([(rds[0], None), (rds[1], None)], ctx=ctx, stats=st)
    runs = ctx.stage_u64(np.array([0, 0, v2.n_chunks, 1, 0, v3.n_chunks], dtype=np.uint64))
    n_out = v2.n_chunks + v3.n_chunks
    ptrs = torch.full((8 * n_out,), 0xAB, dtype=torch.uint8, device=ctx.tdev)
    index = torch.full((40 * 4,), 0xAB, dtype=torch.uint8, device=ctx.tdev)
    store = torch.full((64,), 0xAB, dtype=torch.uint8, device=ctx.tdev)
    dstore = torch.full((64,), 0xAB, dtype=torch.uint8, device=ctx.tdev)
    out6 = (C.c_uint64 * 6)()
    args = (ptrs.data_ptr(), index.data_ptr(), 4, store.data_ptr(), 64, dstore.data_ptr(), 64, out6, ctx.stream)
    rc = ctx.lib.hmse_compose(ctx.h, _desc(rds), 2, runs.data_ptr(), 2, n_out, *args)
    assert rc == _lib.HMSE_E_CAPACITY
    assert list(out6) == [n_out, st["stored_referenced"], want.n_unique, want.store.size, want.n_delta, want.delta_store.size]
    untouched = lambda: all(bool((t == 0xAB).all()) for t in (ptrs, index, store, dstore))  # noqa: E731
    assert untouched()
    bad = ctx.stage_u64(np.array([0, 0, v2.n_chunks, 1, 5, v3.n_chunks], dtype=np.uint64))
    rc = ctx.lib.hmse_compose(ctx.h, _desc(rds), 2, bad.data_ptr(), 2, n_out, *args)
    assert rc == _lib.HMSE_E_INVAL and b"outside" in ctx.lib.hmse_last_error(ctx.h)
    bad = ctx.stage_u64(np.array([2, 0, 1], dtype=np.uint64))
    rc = ctx.lib.hmse_compose(ctx.h, _desc(rds), 2, bad.data_ptr(), 1, 1, *args)
    assert rc == _lib.HMSE_E_INVAL
    rc = ctx.lib.hmse_compose(ctx.h, _desc(rds), 2, runs.data_ptr(), 2, n_out - 1, *args)
    assert rc == _lib.HMSE_E_INVAL and b"add up" in ctx.lib.hmse_last_error(ctx.h)
    torch.cuda.synchronize()
    assert untouched()


def test_launch_count_does_not_depend_on_sources_or_runs(ctx, corpus8):
    from hmse_b200 import archive
    files = _mix(corpus8, 30, 40)
    rd = archive.Reader(_ingest(ctx, files), ctx)
    rng = np.random.default_rng(2)
    counts = []
    for parts in ([(rd, None)], [(rd, None)] * 8, [(rd, rng.integers(0, 40, 10).tolist())],
                  [(rd, rng.integers(0, 40, 100000).tolist())]):
        n0 = ctx.lib.hmse_launch_count(ctx.h)
        archive.compose(parts, ctx=ctx)
        counts.append(ctx.lib.hmse_launch_count(ctx.h) - n0)
    assert len(set(counts)) == 1, counts
