"""Ingest against an existing archive (hmse_compress_known, Ingest.run(known=...), IngestStream.run(known=...)): every
field of the result, and the archive built from it, equals the plain ingest's, for bases that hold a subset of the files,
all of them, none of them, nothing at all, no file table, and deltas (v2, v3), with L4 on the new ingest and with
multi-block streams; which streams were copied equals the CPU reference (tests/known_ref.py), and only the others were
parsed; the snapshot workflow (ingest against the base, build, compose with the base) equals one ingest; a digest whose
stored chunk has another raw length is compressed; streaming runs keep their dedup session; stores past 2^32; bad input
is rejected before anything is written, and a capacity retry packs without compressing again."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from oracle import corpus
from tests import compose_ref, known_ref

pytestmark = pytest.mark.gpu

FIELDS = ("cuts", "digests", "canon", "is_first", "select", "blob", "offsets", "file_chunk", "base", "delta_blob",
          "delta_offsets")


def _run(ctx, files, known=None, l4=False, cdc=None):
    import hmse_b200
    data = np.concatenate(files)
    ing = hmse_b200.Ingest(ctx, cdc or hmse_b200.CDCConfig(), corpus.zdict())
    return ing.run(ctx.stage(data), files=[f.size for f in files], l4=hmse_b200.SimConfig() if l4 else None, known=known)


def _build(ctx, res):
    from hmse_b200 import archive
    return archive.build(res, corpus.zdict(), ctx=ctx)


def _mix(corpus8, seed, n, hi=96 << 10):
    """n files cut from random places of the corpus (overlaps, so chunks repeat across files), some empty."""
    rng = np.random.default_rng(seed)
    files = []
    for _ in range(n):
        size = int(rng.integers(0, hi)) if rng.random() > 0.1 else 0
        a = int(rng.integers(0, corpus8.size - size))
        files.append(corpus8[a:a + size])
    return files


def _same(a, b):
    import torch
    for f in FIELDS:
        x, y = getattr(a, f), getattr(b, f)
        assert (x is None) == (y is None), f
        if x is not None:
            assert torch.equal(x.cpu(), y.cpu()), f
    assert (a.entry, a.id_base) == (b.entry, b.id_base)


def _check_known(ctx, res, base, parse_stats=True):
    """res.known and res.stats against the reference; only the compressed chunks were parsed."""
    buf = getattr(base, "ar", base).tobytes()
    sel = res.select.cpu().numpy()
    cuts = res.cuts.cpu().numpy()
    lens = (cuts - np.concatenate([[0], cuts[:-1]]))[sel]
    want = known_ref.known(buf, res.digests.cpu().numpy()[sel], lens)
    assert np.array_equal(res.known.cpu().numpy(), want)
    clen = np.diff(compose_ref._parse(buf)["upos"])
    assert res.stats == dict(copied=int((want >= 0).sum()), copied_bytes=int(clen[want[want >= 0]].sum()),
                             compressed=int((want < 0).sum()), compressed_raw_bytes=int(lens[want < 0].sum()))
    if parse_stats:
        out4 = (C.c_uint64 * 4)()
        ctx.check(ctx.lib.hmse_compress_stats(ctx.h, out4, None, None))
        assert (int(out4[3]), int(out4[2])) == (res.stats["compressed"], res.stats["compressed_raw_bytes"])
    return want


def _identity(ctx, files, base, l4=False, cdc=None, parse_stats=True):
    plain = _run(ctx, files, l4=l4, cdc=cdc)
    got = _run(ctx, files, known=base, l4=l4, cdc=cdc)
    _same(got, plain)
    assert plain.known is None and plain.stats is None
    assert _build(ctx, got).tobytes() == _build(ctx, plain).tobytes()
    return _check_known(ctx, got, base, parse_stats)


@pytest.fixture(scope="module")
def new_files(corpus8):
    return _mix(corpus8, 1, 70)


def test_base_with_a_subset_of_the_files(ctx, new_files):
    base = _build(ctx, _run(ctx, new_files[::2]))
    kn = _identity(ctx, new_files, base)
    assert 0 < (kn >= 0).sum() < kn.size


def test_base_with_the_same_files_copies_every_stream(ctx, new_files):
    from hmse_b200 import archive
    base = _build(ctx, _run(ctx, new_files))
    kn = _identity(ctx, new_files, archive.Reader(base, ctx))
    assert (kn >= 0).all() and np.array_equal(kn, np.arange(kn.size))


def test_disjoint_base_copies_nothing(ctx, new_files):
    import torch
    g = torch.Generator(device=ctx.tdev).manual_seed(3)
    noise = torch.randint(0, 256, (3 << 20,), dtype=torch.uint8, device=ctx.tdev, generator=g).cpu().numpy()
    base = _build(ctx, _run(ctx, [noise[:1 << 20], noise[1 << 20:]]))
    assert (_identity(ctx, new_files, base) < 0).all()


def test_empty_base(ctx, new_files):
    from hmse_b200 import archive
    u8 = np.uint8
    empty = archive.Archive(corpus.zdict(), np.zeros((0, 40), u8), np.zeros((0, 8), u8), np.zeros(0, u8), 0)
    assert (_identity(ctx, new_files, empty, parse_stats=False) < 0).all()


def test_v1_base(ctx, corpus8, new_files):
    import hmse_b200
    zd = corpus.zdict()
    v1 = _build(ctx, hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(corpus8[:4 << 20])))
    assert v1.file_chunk is None
    kn = _identity(ctx, new_files, v1)
    assert 0 < (kn >= 0).sum() < kn.size


@pytest.fixture(scope="module")
def delta_bases(ctx, corpus8):
    import hmse_b200
    d2 = np.concatenate([corpus8[:6 << 20], corpus8[2 << 20:3 << 20]])
    v2 = _build(ctx, hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), corpus.zdict()).run(ctx.stage(d2), l4=hmse_b200.SimConfig()))
    assert v2.n_delta > 20 and v2.file_chunk is None
    rng = np.random.default_rng(4)
    sizes = rng.integers(0, 256 << 10, 40)
    sizes[-1] = 0
    sizes[-1] = d2.size - int(sizes.sum())
    off = np.concatenate([[0], np.cumsum(sizes)])
    files = [d2[off[f]:off[f + 1]] for f in range(40)]
    v3 = _build(ctx, _run(ctx, files, l4=True))
    assert v3.n_delta > 20 and v3.file_chunk is not None
    return v2, v3, files


@pytest.mark.parametrize("which", ["v2", "v3"])
def test_bases_with_deltas(ctx, delta_bases, new_files, which):
    v2, v3, files = delta_bases
    base = v2 if which == "v2" else v3
    kn = _identity(ctx, new_files, base)
    assert 0 < (kn >= 0).sum() < kn.size
    # the base's own files again, with L4 on the new ingest: delta targets are first occurrences with no index entry
    kn = _identity(ctx, files[::-1], base, l4=True)
    assert 0 < (kn >= 0).sum() < kn.size


def test_multi_block_streams(ctx, corpus8):
    import hmse_b200
    cdc = hmse_b200.CDCConfig(16 << 10, 32 << 10, 64 << 10)
    files = _mix(corpus8, 5, 40, hi=512 << 10)
    base = _build(ctx, _run(ctx, files[:25], cdc=cdc))
    kn = _identity(ctx, files, base, cdc=cdc, parse_stats=False)
    plain = _run(ctx, files, cdc=cdc)
    cuts = plain.cuts.cpu().numpy()
    lens = (cuts - np.concatenate([[0], cuts[:-1]]))[plain.select.cpu().numpy()]
    assert (lens[kn >= 0] > 32 << 10).sum() > 10     # streams of several blocks were copied
    assert (kn < 0).sum() > 0


def test_snapshot_workflow(ctx, corpus8):
    from hmse_b200 import archive
    old = _mix(corpus8, 11, 50)
    new = [f.copy() for f in old[10:]] + _mix(corpus8, 12, 20)
    for f in new[::4]:
        if f.size:
            f[f.size // 2] ^= 0x41
    base = _build(ctx, _run(ctx, old))
    rd = archive.Reader(base, ctx)
    snap = _build(ctx, _run(ctx, new, known=rd))
    st = {}
    got = archive.compose([(rd, None), (snap, None)], ctx=ctx, stats=st)
    assert got.tobytes() == _build(ctx, _run(ctx, old + new)).tobytes()
    assert st["deduplicated"] > 0


def test_length_check(ctx, new_files):
    plain = _run(ctx, new_files)
    base = _build(ctx, _run(ctx, new_files[::2]))
    sel = plain.select.cpu().numpy()
    cuts = plain.cuts.cpu().numpy()
    lens = (cuts - np.concatenate([[0], cuts[:-1]]))[sel]
    dg = plain.digests.cpu().numpy()[sel]
    kn = known_ref.known(base.tobytes(), dg, lens)
    _, ulen = known_ref.slot_lengths(base.tobytes())
    k = int(np.flatnonzero(kn < 0)[0])
    s = int(np.flatnonzero(ulen != lens[k])[0])
    index = base.index.copy()
    index[s, :32] = dg[k]
    bad = dataclasses.replace(base, index=index)
    got = _run(ctx, new_files, known=bad)
    _same(got, plain)
    assert int(got.known[k]) == -1
    _check_known(ctx, got, bad)


def test_stream_runs_keep_their_dedup_session(ctx, corpus8):
    import torch
    import hmse_b200
    from hmse_b200 import archive
    zd = corpus.zdict()
    data = np.concatenate([corpus8[:3 << 20], corpus8[5 << 20:7 << 20], corpus8[1 << 20:2 << 20]])
    base = _build(ctx, _run(ctx, [corpus8[2 << 20:6 << 20]]))
    host = torch.from_numpy(data).pin_memory()
    st = hmse_b200.IngestStream(ctx, hmse_b200.CDCConfig(), zd, piece_bytes=1 << 20)
    assert len(st.schedule(data.size)) > 4
    plain = st.run(host)
    plain = dataclasses.replace(plain, cuts=plain.cuts.clone(), digests=plain.digests.clone(), canon=plain.canon.clone(),
                                offsets=plain.offsets.clone(), blob=plain.blob.clone())
    got = st.run(host, known=archive.Reader(base, ctx))
    for f in ("cuts", "digests", "canon", "offsets", "blob"):
        assert torch.equal(getattr(got, f), getattr(plain, f)), f
    one = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(data))
    assert torch.equal(got.blob, one.blob.cpu()) and torch.equal(got.canon, one.canon.cpu())
    sel = got.select.numpy()
    cuts = got.cuts.numpy()
    lens = (cuts - np.concatenate([[0], cuts[:-1]]))[sel]
    want = known_ref.known(base.tobytes(), got.digests.numpy()[sel], lens)
    assert np.array_equal(got.known.numpy(), want)
    assert 0 < got.stats["copied"] == int((want >= 0).sum()) < sel.size
    assert got.stats["compressed"] == int((want < 0).sum())


def test_store_past_2_32(ctx):
    import torch
    import hmse_b200
    from hmse_b200 import archive
    zd = corpus.zdict()
    g = torch.Generator(device=ctx.tdev).manual_seed(5)
    n = 2_200_000_000
    srcs = []
    for _ in range(2):
        d = torch.randint(0, 256, (n,), dtype=torch.uint8, device=ctx.tdev, generator=g)
        srcs.append(_build(ctx, hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(d), files=[n])))
    tail = d[n - (64 << 20):]
    del d
    base = archive.compose([(srcs[0], None), (srcs[1], None)], ctx=ctx)
    del srcs
    assert base.store.size > (1 << 32)
    rd = archive.Reader(base, ctx)
    fresh = torch.randint(0, 256, (8 << 20,), dtype=torch.uint8, device=ctx.tdev, generator=g)
    new = torch.cat([fresh[:4 << 20], tail, fresh[4 << 20:]])
    ing = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd)
    plain = ing.run(ctx.stage(new), files=[new.numel()])
    got = ing.run(ctx.stage(new), files=[new.numel()], known=rd)
    _same(got, plain)
    upos = np.concatenate([[0], np.cumsum(base.index[:, 36:38].copy().view("<u2").reshape(-1).astype(np.int64))])
    kn = got.known.cpu().numpy()
    assert (upos[kn[kn >= 0]] > (1 << 32)).sum() > 1000
    assert (kn < 0).sum() > 500


def _desc(rd, m=None):
    d = rd.src()
    if m is not None:
        d.m = m
    return d


def test_errors(ctx, new_files):
    import torch
    import hmse_b200
    from hmse_b200 import _lib, archive
    zd = corpus.zdict()
    base = _build(ctx, _run(ctx, new_files[::2]))
    with pytest.raises(ValueError, match="dictionary"):
        _run(ctx, new_files, known=dataclasses.replace(base, zdict=zd[:-1]))
    with pytest.raises(ValueError, match="compress"):
        hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(np.concatenate(new_files)), compress=False, known=base)

    rd = archive.Reader(base, ctx)
    plain = _run(ctx, new_files)
    data = ctx.stage(np.concatenate(new_files))
    m = plain.select.numel()
    dz = ctx.stage(zd)
    offs = torch.full((m + 1,), -7, dtype=torch.int64, device=ctx.tdev)
    kn = torch.full((m,), -7, dtype=torch.int64, device=ctx.tdev)
    out = torch.full((plain.blob.numel() + 64,), 0xAB, dtype=torch.uint8, device=ctx.tdev)
    total, st4 = C.c_uint64(0), (C.c_uint64 * 4)()

    def call(src, out_ptr, cap, zp=dz.data_ptr(), zl=len(zd), cuts=plain.cuts.data_ptr(), offp=offs.data_ptr()):
        return ctx.lib.hmse_compress_known(ctx.h, C.byref(src) if src is not None else None, data.data_ptr(), 0, cuts,
                                           plain.digests.data_ptr(), plain.select.data_ptr(), m, zp, zl, 6, out_ptr, cap, offp,
                                           C.byref(total), kn.data_ptr(), st4, ctx.stream)

    def untouched():
        torch.cuda.synchronize()
        return bool((offs == -7).all()) and bool((kn == -7).all()) and bool((out == 0xAB).all())

    assert call(_desc(rd, rd.m - 1), out.data_ptr(), out.numel()) == _lib.HMSE_E_INVAL
    assert b"layout" in ctx.lib.hmse_last_error(ctx.h) and untouched()
    assert call(_desc(rd), out.data_ptr(), out.numel(), zl=len(zd) - 1) == _lib.HMSE_E_INVAL
    assert b"dictionary" in ctx.lib.hmse_last_error(ctx.h) and untouched()
    assert call(_desc(rd), out.data_ptr(), out.numel(), zp=None, zl=0) == _lib.HMSE_E_INVAL and untouched()
    assert call(None, out.data_ptr(), out.numel()) == _lib.HMSE_E_INVAL and untouched()
    assert call(_desc(rd), out.data_ptr(), out.numel(), offp=None) == _lib.HMSE_E_INVAL and untouched()
    assert call(_desc(rd), out.data_ptr(), out.numel(), cuts=plain.cuts.data_ptr() + 4) == _lib.HMSE_E_INVAL and untouched()
    assert call(_desc(rd), out.data_ptr(), out.numel(), offp=offs.data_ptr() + 4) == _lib.HMSE_E_INVAL and untouched()

    # too small: the size needed comes back, and the pack writes the planned streams without compressing anything
    assert call(_desc(rd), out.data_ptr(), 100) == _lib.HMSE_E_CAPACITY
    assert total.value == plain.blob.numel()
    torch.cuda.synchronize()
    assert bool((out == 0xAB).all())
    n0 = ctx.lib.hmse_launch_count(ctx.h)
    ctx.check(ctx.lib.hmse_compress_known_pack(ctx.h, offs.data_ptr(), m, out.data_ptr(), out.numel(), ctx.stream))
    assert ctx.lib.hmse_launch_count(ctx.h) - n0 == 1
    torch.cuda.synchronize()
    assert torch.equal(out[:total.value], plain.blob) and torch.equal(offs, plain.offsets)
    # sizes only, then the pack
    out.fill_(0xAB)
    assert call(_desc(rd), None, 0) == 0 and total.value == plain.blob.numel()
    n0 = ctx.lib.hmse_launch_count(ctx.h)
    ctx.check(ctx.lib.hmse_compress_known_pack(ctx.h, offs.data_ptr(), m, out.data_ptr(), out.numel(), ctx.stream))
    assert ctx.lib.hmse_launch_count(ctx.h) - n0 == 1
    torch.cuda.synchronize()
    assert torch.equal(out[:total.value], plain.blob)
    # a plain hmse_compress in between overwrites the staged streams: the plan is gone
    ctx.compress(data, plain.cuts, plain.select[:5], dz)
    assert ctx.lib.hmse_compress_known_pack(ctx.h, offs.data_ptr(), m, out.data_ptr(), out.numel(), ctx.stream) == _lib.HMSE_E_INVAL
