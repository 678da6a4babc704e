"""CPU tests of bench.py's command line and of what --dump-outputs writes (the dump writers on results in host memory)."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ingest_result(n, m, nb):
    from hmse_b200.ingest import IngestResult
    g = torch.Generator().manual_seed(n)
    cuts = torch.cumsum(torch.randint(2048, 32768, (n,), generator=g), 0) + (1 << 40)     # above 2^32, below 2^53
    digests = torch.randint(0, 256, (n, 32), dtype=torch.uint8, generator=g)
    canon = torch.randint(0, n, (n,), generator=g)
    first = torch.rand(n, generator=g) < 0.7
    select = torch.sort(torch.randperm(n, generator=g)[:m]).values
    blob = torch.randint(0, 256, (nb,), dtype=torch.uint8, generator=g)
    offsets = torch.cat([torch.zeros(1, dtype=torch.int64), torch.sort(torch.randint(0, nb, (m,), generator=g)).values])
    return IngestResult(cuts, digests, canon, first, select, blob, offsets, entry=123, id_base=7)


def _similarity_step(n, t):
    g = torch.Generator().manual_seed(n)
    full = lambda *shape: torch.randint(-(1 << 63), (1 << 63) - 1, shape, generator=g)    # noqa: E731  (every bit pattern)
    return {"cuts": torch.cumsum(torch.randint(2048, 32768, (n,), generator=g), 0), "entry": 5, "id_base": 9, "n_total": 4 * n,
            "sig": full(n, 128).to(torch.int32), "keys": full(n, 32), "band": torch.randint(0, 32, (t,), generator=g).to(torch.int32),
            "key": full(t), "ids": torch.randint(0, 4 * n, (t,), generator=g)}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def _dump_bytes(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def test_ingest_dump_exact_repeatable_and_under_64_mb_for_every_world(tmp_path):
    import bench
    n, nb = 3 << 17, (1 << 20) + 12345
    res = _ingest_result(n, n // 2, nb)
    bench.dump_ingest(str(tmp_path / "a"), res, 0, 1)
    bench.dump_ingest(str(tmp_path / "b"), _ingest_result(n, n // 2, nb), 0, 1)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    whole = {"cuts": res.cuts, "digests": res.digests, "canon": res.canon, "is_first": res.is_first, "select": res.select,
             "offsets": res.offsets, "blob": res.blob}
    assert sorted(a) == sorted(list(whole) + ["counts"])
    for name, t in whole.items():
        rows = bench.dump_rows(t.shape[0], (1 << 20) if name == "blob" else (1 << 17))
        assert rows.size < t.shape[0] and np.array_equal(a[name], t.numpy()[rows].astype(a[name].dtype)), name
    assert a["counts"].tolist() == [123, 7, n, n // 2, nb]
    # every rank's files in one directory: the dump as a whole stays under 64 MB
    for world in (1, 2, 8):
        d = tmp_path / ("w%d" % world)
        for rank in range(world):
            bench.dump_ingest(str(d), res, rank, world)
        assert len(os.listdir(d)) == 8 * world and _dump_bytes(d) <= 64_000_000, (world, _dump_bytes(d))
    # a result below the limits is written whole
    small = _ingest_result(1000, 400, 5000)
    bench.dump_ingest(str(tmp_path / "s"), small, 1, 2)
    s = _load(tmp_path / "s")
    assert sorted(s) == sorted(k + ".rank1" for k in list(whole) + ["counts"])
    assert np.array_equal(s["cuts.rank1"], small.cuts.numpy().astype(np.float64))
    assert np.array_equal(s["digests.rank1"], small.digests.numpy().astype(np.float32))
    assert np.array_equal(s["blob.rank1"], small.blob.numpy().astype(np.float32))


def test_similarity_dump_exact_and_under_64_mb_for_every_world(tmp_path):
    import bench
    n, t = 3 << 14, 3 << 17
    out = _similarity_step(n, t)
    bench.dump_similarity(str(tmp_path / "a"), out, 0, 1)
    a = _load(tmp_path / "a")
    assert sorted(a) == ["band", "counts", "cuts", "ids", "key", "keys", "sig"]
    assert all(v.dtype == np.float64 for v in a.values())
    r, rt = bench.dump_rows(n, 1 << 14), bench.dump_rows(t, 1 << 17)
    assert np.array_equal(a["sig"], out["sig"].numpy()[r].view(np.uint32).astype(np.float64))
    for name, rows in (("keys", r), ("key", rt)):
        u = out[name].numpy()[rows].view(np.uint64)
        got = a[name].astype(np.uint64)
        assert got.shape == u.shape + (2,) and np.array_equal((got[..., 0] << np.uint64(32)) | got[..., 1], u), name
    assert np.array_equal(a["band"], out["band"].numpy()[rt].astype(np.float64))
    assert np.array_equal(a["ids"], out["ids"].numpy()[rt].astype(np.float64))
    assert a["counts"].tolist() == [5, 9, 4 * n, n, t]
    for world in (1, 2, 8):
        d = tmp_path / ("w%d" % world)
        for rank in range(world):
            bench.dump_similarity(str(d), out, rank, world)
        assert len(os.listdir(d)) == 7 * world and _dump_bytes(d) <= 64_000_000, (world, _dump_bytes(d))
    # a rank that owns no band
    bench.dump_similarity(str(tmp_path / "e"), dict(out, band=None, key=None, ids=None), 1, 2)
    e = _load(tmp_path / "e")
    assert e["band.rank1"].size == 0 and e["key.rank1"].shape == (0, 2) and e["counts.rank1"][4] == 0


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert r.returncode == 2 and "--steps" in r.stderr
