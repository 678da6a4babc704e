"""Random-access reads (archive.Reader, hmse_read) on the seed-42 device corpus ingested into an archive.

Records: Reader open time; one batch each of 10^4, 10^5 and 10^6 random 4 KiB reads and 10^5 random 64 KiB reads
(reads/s, GB/s requested, GB/s inflated, amplification = raw bytes inflated / bytes requested, and the split between
plan, inflate, delta and copy from the hmse timers); the same 10^4 reads made one call per range; and the whole-stream
restore at this commit next to the restore of another archive.py (--parent, e.g. the previous commit's), alternated in
the same process.  Records the GPU name and power limit, writes one JSON (default profiles/read_bench.json) and fails
without a GPU.  `python tools/read_bench.py [--gb 10] [--parent old_archive.py]`."""
from __future__ import annotations

import argparse
import ctypes as C
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

T_INFLATE, T_DELTA, T_READ_PLAN, T_READ_COPY = 8, 9, 11, 12


def gpu_facts():
    import torch
    facts = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        facts["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else None
    except (OSError, subprocess.SubprocessError):
        facts["power_limit_and_max_sm_clock"] = None
    return facts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=10.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parent", default=None, help="an archive.py whose restore() is timed next to this one")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "read_bench.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("read_bench.py needs a CUDA device")
    import hmse_b200
    from hmse_b200 import archive
    from hmse_b200 import corpus as pc
    ctx = hmse_b200.Context(0)
    lib = ctx.lib
    n = int(a.gb * 1e9) & ~15
    zd = pc.zdict()
    t0 = time.perf_counter()
    d = pc.DeviceCorpus(ctx).generate(n)
    r = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), ctx.stage(zd)).run(d[:n])
    ar = archive.build(r, zd, ctx=ctx)
    del r
    torch.cuda.synchronize()
    res = dict(gpu_facts(), raw_bytes=ar.raw_bytes, chunks=ar.n_chunks, stored_chunks=ar.n_unique, store_bytes=int(ar.store.size),
               build_s=round(time.perf_counter() - t0, 1), batches={})
    print(json.dumps(res), flush=True)
    opens = []
    for _ in range(a.reps):
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        rd = archive.Reader(ar, ctx)
        torch.cuda.synchronize()
        opens.append((time.perf_counter() - w0) * 1e3)
    res["open_ms"] = [round(x, 1) for x in opens]
    # the open without the host-to-device copies: hmse_read_open alone on the staged records
    idx, ptr = ctx.stage(ar.index.reshape(-1)), ctx.stage(ar.pointers.reshape(-1))
    ko = []
    for _ in range(a.reps):
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        ctx.check(lib.hmse_read_open(ctx.h, idx.data_ptr(), rd.m, ptr.data_ptr(), rd.n, int(ar.store.size), None, 0, 0,
                                     rd.raw_bytes, rd.zd.data_ptr(), len(zd), rd.layout.data_ptr(), rd.layout.numel(), ctx.stream))
        ko.append((time.perf_counter() - w0) * 1e3)
    res["open_device_ms"] = [round(x, 2) for x in ko]
    raw = ar.raw_bytes
    rng = np.random.default_rng(42)

    def timed_read(off, ln):
        lib.hmse_timing(ctx.h, 1)
        st = {}
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        rd.read(off, ln, device_out=True, stats=st)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - w0) * 1e3
        f = C.c_float(0)
        split = {}
        for name, tid in (("plan", T_READ_PLAN), ("inflate", T_INFLATE), ("delta", T_DELTA), ("copy", T_READ_COPY)):
            split[name] = round(f.value, 3) if lib.hmse_timing_ms(ctx.h, tid, C.byref(f)) == 0 else None
        lib.hmse_timing(ctx.h, 0)
        return wall, split, st

    for R, size in ((10_000, 4096), (100_000, 4096), (1_000_000, 4096), (100_000, 65536)):
        off = rng.integers(0, raw - size, R, dtype=np.int64)
        ln = np.full(R, size, dtype=np.int64)
        timed_read(off, ln)                       # warm-up: scratch at its size
        runs = [timed_read(off, ln) for _ in range(a.reps)]
        wall = statistics.median(x[0] for x in runs)
        st = runs[0][2]
        req = R * size
        rec = {"ranges": R, "bytes": size, "call_ms": [round(x[0], 2) for x in runs], "reads_per_s": int(R / (wall * 1e-3)),
               "GB_per_s_requested": round(req / (wall * 1e-3) / 1e9, 2),
               "GB_per_s_inflated": round(st["inflated_bytes"] / (wall * 1e-3) / 1e9, 2),
               "amplification": round(st["inflated_bytes"] / req, 3), "streams_inflated": st["inflated"],
               "split_ms": runs[-1][1]}
        sp = rec["split_ms"]
        rec["plan_share"] = round(sp["plan"] / wall, 3) if sp["plan"] is not None else None
        res["batches"]["%dx%d" % (R, size)] = rec
        print(json.dumps({"%dx%d" % (R, size): rec}), flush=True)
    # the same 10^4 reads, one call per range
    off = rng.integers(0, raw - 4096, 10_000, dtype=np.int64)
    rd.read(off[:10], np.full(10, 4096), device_out=True)
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    for o in off:
        rd.read([int(o)], [4096], device_out=True)
    torch.cuda.synchronize()
    one = (time.perf_counter() - w0) * 1e3
    res["one_call_per_range_10000x4096"] = {"ms": round(one, 1), "reads_per_s": int(10_000 / (one * 1e-3))}
    print(json.dumps(res["one_call_per_range_10000x4096"]), flush=True)
    # whole-stream restore, this commit against --parent, alternated
    del rd
    torch.cuda.empty_cache()
    impls = {"this": archive.restore}
    if a.parent:
        spec = importlib.util.spec_from_file_location("hmse_b200._parent_archive", a.parent)
        mod = importlib.util.module_from_spec(spec)
        sys.modules[spec.name] = mod
        spec.loader.exec_module(mod)
        impls["parent"] = mod.restore
    want = None
    times = {k: [] for k in impls}
    for it in range(a.reps + 1):
        for k, fn in impls.items():
            torch.cuda.synchronize()
            w0 = time.perf_counter()
            out = fn(ar, ctx=ctx)
            torch.cuda.synchronize()
            if it:
                times[k].append((time.perf_counter() - w0) * 1e3)
            if want is None:
                want = d[:n].cpu().numpy()
            assert out.size == n and np.array_equal(out, want), k
            del out
    res["restore_whole_stream_ms"] = {k: [round(x, 1) for x in v] for k, v in times.items()}
    res["restore_median_ms"] = {k: round(statistics.median(v), 1) for k, v in times.items()}
    print(json.dumps({"restore": res["restore_whole_stream_ms"]}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
