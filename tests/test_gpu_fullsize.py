"""Parity against the oracle at the sizes BASELINE.json quotes (SURVEY.md section 7, hard part 4): the 1 GiB seed-42
base of config 1, and a stream longer than 4 GiB where a 32-bit offset anywhere in scan, resolve, digest, dedup or pack
would show.  The bytes come from the device generator (bit-identical to oracle/corpus.py: checked here on a prefix and on
windows, and in tests/test_gpu_corpus_lsh.py), are copied to the host, and the oracle (chunk_c = Algorithm 1 in C,
hashlib SHA-256, the dict dedup) runs over ALL of them: the cut list, every digest, canon and is_first must be equal.
Determinism criterion: VALIDATION_METHODS.md:190-194 of the HMSE spec."""
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _oracle_all(host, cfg):
    import oracle
    cuts = oracle.chunk_c(host, cfg)
    dg = oracle.digest_mt(host, cuts)
    canon, first = oracle.dedup(dg)
    return cuts, dg, canon, first


def _anchor_generator(gen, host, offsets, span=1 << 20):
    """The device generator's bytes equal the oracle generator's near each of `offsets`: the article that starts at or
    after the offset is located through the generator's article table and re-rendered from there by oracle/corpus.py."""
    from oracle import corpus
    art = gen._offs.cpu().numpy()
    for o in offsets:
        a = int(np.searchsorted(art, o))
        lo = int(art[a])
        assert lo + span <= host.size
        want = corpus.generate(span, first_article=a)
        assert np.array_equal(host[lo:lo + span], want), "device corpus differs from oracle/corpus.py at byte %d (article %d)" % (lo, a)


def _check_streams(res, host, cuts, sel, zd, sample):
    """`sample` of the compressed streams through stock zlib with the preset dictionary (the GPU read path checks all)."""
    blob = res.blob.cpu().numpy()
    offs = res.offsets.cpu().numpy()
    starts = np.concatenate([[0], cuts[:-1]]).astype(np.int64)
    for k in sample:
        j = int(sel[k])
        do = zlib.decompressobj(zdict=zd) if zd else zlib.decompressobj()
        raw = do.decompress(blob[offs[k]:offs[k + 1]].tobytes()) + do.flush()
        assert raw == host[starts[j]:int(cuts[j])].tobytes(), "stream %d (chunk %d) does not inflate to its chunk" % (k, j)


def test_config1_one_gib_equals_the_oracle(ctx):
    import torch
    import hmse_b200
    from hmse_b200 import corpus as pc
    from oracle import corpus
    n = 1 << 30
    cfg = hmse_b200.CDCConfig()
    zdb = pc.zdict()
    assert zdb == corpus.zdict()
    zd = ctx.stage(zdb)
    gen = pc.DeviceCorpus(ctx)
    d = gen.generate(n)
    res = hmse_b200.Ingest(ctx, cfg, zd).run(d)
    torch.cuda.synchronize()
    host = d.cpu().numpy()
    _anchor_generator(gen, host, [0, 511 << 20, n - (3 << 20)])
    want_cuts, want_dg, want_canon, want_first = _oracle_all(host, cfg)
    cuts = res.cuts.cpu().numpy().view(np.uint64)
    assert cuts.size == want_cuts.size and np.array_equal(cuts, want_cuts)
    dg = res.digests.cpu().numpy()
    # order-independent aggregates first (what a sharded run can compare cheaply), then every row
    assert np.array_equal(np.bitwise_xor.reduce(dg.view(np.uint64), axis=0), np.bitwise_xor.reduce(want_dg.view(np.uint64), axis=0))
    assert np.array_equal(dg.view(np.uint64).sum(axis=0), want_dg.view(np.uint64).sum(axis=0))
    assert np.array_equal(dg, want_dg)
    assert np.array_equal(res.canon.cpu().numpy(), want_canon)
    assert np.array_equal(res.is_first.cpu().numpy(), want_first)
    sel = res.select.cpu().numpy()
    assert np.array_equal(sel, np.flatnonzero(want_first)) and int(want_first.sum()) < want_first.size
    bad, same = hmse_b200.verify_roundtrip(ctx, res, zd)
    assert bad == 0 and same
    rng = np.random.default_rng(1)
    _check_streams(res, host, cuts, sel, zdb, rng.choice(sel.size, 3000, replace=False))
    # size against zlib level 6 on a sample of the same chunks (config 3's bar, on CDC chunks)
    import oracle
    pick = np.sort(rng.choice(sel.size, 4000, replace=False))
    zb, _ = oracle.compress(host, want_cuts, sel[pick], zdb)
    offs = res.offsets.cpu().numpy()
    ours = int((offs[pick + 1] - offs[pick]).sum())
    assert zb.size / ours >= 0.98


def test_stream_longer_than_4gib_equals_the_oracle(ctx):
    """5 GB in one buffer: offsets cross 2^32 inside the stream, inside the resolve segments and inside the DEFLATE
    stage.  Everything is compared, not windows; the streaming front end (host pieces) must give the same."""
    import torch
    import hmse_b200
    from hmse_b200 import corpus as pc
    n = 5_000_000_000 - (5_000_000_000 % 16)
    assert n > (1 << 32) + (256 << 20)
    cfg = hmse_b200.CDCConfig()
    zdb = pc.zdict()
    zd = ctx.stage(zdb)
    gen = pc.DeviceCorpus(ctx)
    d = gen.generate(n)
    res = hmse_b200.Ingest(ctx, cfg, zd).run(d)
    torch.cuda.synchronize()
    host_t = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    host_t.copy_(d)
    host = host_t.numpy()
    _anchor_generator(gen, host, [(1 << 32) - (2 << 20), (1 << 32) + (5 << 20), n - (3 << 20)])
    want_cuts, want_dg, want_canon, want_first = _oracle_all(host, cfg)
    cuts = res.cuts.cpu().numpy().view(np.uint64)
    assert int(cuts[-1]) == n and (cuts > np.uint64(1 << 32)).sum() > 50000
    assert cuts.size == want_cuts.size and np.array_equal(cuts, want_cuts)
    assert np.array_equal(res.digests.cpu().numpy(), want_dg)
    assert np.array_equal(res.canon.cpu().numpy(), want_canon) and np.array_equal(res.is_first.cpu().numpy(), want_first)
    sel = res.select.cpu().numpy()
    bad, same = hmse_b200.verify_roundtrip(ctx, res, zd)
    assert bad == 0 and same
    # streams of chunks on both sides of 2^32 through stock zlib
    k32 = int(np.searchsorted(cuts[sel], np.uint64(1 << 32)))
    _check_streams(res, host, cuts, sel, zdb, list(range(max(0, k32 - 300), min(sel.size, k32 + 300))) + [0, sel.size - 1])
    want_blob_bytes = int(res.blob.numel())
    want_offs = res.offsets.cpu().numpy()
    del res, d
    torch.cuda.empty_cache()
    # the same stream through the host-to-host front end in 1 GiB pieces (piece boundaries, absolute offsets > 2^32)
    hres = hmse_b200.IngestStream(ctx, cfg, zd, piece_bytes=1 << 30).run(host_t)
    assert np.array_equal(hres.cuts.numpy().view(np.uint64), want_cuts)
    assert np.array_equal(hres.digests.numpy(), want_dg)
    assert np.array_equal(hres.canon.numpy(), want_canon)
    assert int(hres.blob.numel()) == want_blob_bytes and np.array_equal(hres.offsets.numpy(), want_offs)
