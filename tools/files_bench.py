"""Many files in one call: hmse_chunk_files next to hmse_chunk on the same bytes, and Ingest.run with and without files.

Renders `--gb` GB of the seed-42 corpus on the device and splits it by seeded file-size mixes:
  one_file        the whole buffer as one file (must match hmse_chunk within run-to-run spread)
  lognormal_16k   log-normal sizes, median 16 KiB (sigma 1.2)
  lognormal_2k    log-normal sizes, median 2 KiB (sigma 1.2): millions of files, about half shorter than min_size
  files_64m       64 MiB files
For each mix: HMSE_T_SCAN / HMSE_T_RESOLVE of hmse_chunk_files and of hmse_chunk, alternated after a warm-up; chunk
count and chunks per second; device-resident Ingest.run time with and without files; unique chunks and stored bytes.
Records the GPU name and power limit, writes one JSON (default profiles/files_bench.json) and fails without a GPU.
    python tools/files_bench.py [--gb 10] [--reps 5] [--out profiles/files_bench.json]"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_facts():
    import torch
    facts = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        facts["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else None
    except (OSError, subprocess.TimeoutExpired, IndexError):
        facts["power_limit_and_max_sm_clock"] = None
    return facts


def mixes(n: int):
    rng = np.random.default_rng(42)

    def lognormal(median):
        out, total = [], 0
        while total < n:
            s = np.maximum(rng.lognormal(np.log(median), 1.2, 1 << 20).astype(np.int64), 0)
            out.append(s)
            total += int(s.sum())
        s = np.concatenate(out)
        c = np.cumsum(s)
        k = int(np.searchsorted(c, n))
        s = s[:k + 1].copy()
        s[-1] = n - (int(c[k - 1]) if k else 0)
        return s

    big = 64 << 20
    return {"one_file": np.array([n], dtype=np.int64),
            "lognormal_16k": lognormal(16 << 10),
            "lognormal_2k": lognormal(2 << 10),
            "files_64m": np.array([big] * (n // big) + ([n % big] if n % big else []), dtype=np.int64)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=10.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ingest-reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "files_bench.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("files_bench.py needs a CUDA device")
    import hmse_b200
    from hmse_b200 import corpus as pc
    ctx = hmse_b200.Context(0)
    lib = ctx.lib
    n = int(a.gb * 1e9) & ~15
    cfg = hmse_b200.CDCConfig()
    t0 = time.perf_counter()
    d = pc.DeviceCorpus(ctx).generate(n)
    torch.cuda.synchronize()
    result = dict(gpu_facts(), bytes=n, cdc=[cfg.min_size, cfg.avg_size, cfg.max_size], reps=a.reps,
                  render_s=round(time.perf_counter() - t0, 2), mixes={})
    zd = ctx.stage(pc.zdict())
    cap = n // cfg.min_size + 2

    def timed(fn):
        lib.hmse_timing(ctx.h, 1)
        w0 = time.perf_counter()
        out = fn()
        wall = (time.perf_counter() - w0) * 1e3
        f = C.c_float(0)
        ms = []
        for tid in (0, 1):
            ctx.check(lib.hmse_timing_ms(ctx.h, tid, C.byref(f)))
            ms.append(f.value)
        lib.hmse_timing(ctx.h, 0)
        return out, ms[0], ms[1], wall

    cuts1 = ctx.empty(cap, torch.int64)
    nc = C.c_uint64(0)

    def single():
        ctx.check(lib.hmse_chunk(ctx.h, d.data_ptr(), n, C.byref(ctx.cdc_struct(cfg)), cuts1.data_ptr(), cap, C.byref(nc),
                                 ctx.stream))
        return nc.value

    for name, sizes in mixes(n).items():
        off = torch.from_numpy(np.concatenate([[0], np.cumsum(sizes)])).to(ctx.tdev)
        files = lambda: ctx.chunk_files(d, off, cfg)[0].numel()  # noqa: E731
        files()
        single()                                        # warm-up of both, every scratch slot at its size
        rec = {"files": int(sizes.size), "files_below_min_size": int((sizes < cfg.min_size).sum()),
               "median_size": float(np.median(sizes)), "mean_size": float(sizes.mean())}
        tf, ts = [], []
        for _ in range(a.reps):
            tf.append(timed(files))
            ts.append(timed(single))
        rounds = lib.hmse_chunk_last_rounds(ctx.h)
        med = lambda xs, k: statistics.median(x[k] for x in xs)  # noqa: E731
        lo = lambda xs, k: min(x[k] for x in xs)  # noqa: E731
        for key, xs in (("chunk_files", tf), ("chunk", ts)):
            rec[key] = {"chunks": int(xs[0][0]), "scan_ms_median": med(xs, 1), "scan_ms_min": lo(xs, 1),
                        "resolve_ms_median": med(xs, 2), "resolve_ms_min": lo(xs, 2), "call_ms_median": med(xs, 3),
                        "resolve_ms_all": [round(x[2], 4) for x in xs],
                        "chunks_per_s": int(xs[0][0] / ((med(xs, 1) + med(xs, 2)) * 1e-3))}
        rec["chunk_rounds_last"] = int(rounds)
        rec["resolve_ratio_files_over_chunk"] = rec["chunk_files"]["resolve_ms_median"] / rec["chunk"]["resolve_ms_median"]
        # device-resident ingest (CDC, SHA-256, dedup, DEFLATE of first occurrences), alternated
        ing = hmse_b200.Ingest(ctx, cfg, zd)
        sz_dev = torch.from_numpy(sizes).to(ctx.tdev)
        runs = {"with_files": [], "without_files": []}
        outs = {}
        for it in range(a.ingest_reps + 1):
            for key, kw in (("with_files", {"files": sz_dev}), ("without_files", {})):
                torch.cuda.synchronize()
                w0 = time.perf_counter()
                r = ing.run(d, **kw)
                torch.cuda.synchronize()
                if it:
                    runs[key].append((time.perf_counter() - w0) * 1e3)
                outs[key] = (r.n_chunks, int(r.select.numel()), int(r.blob.numel()))
                del r
        for key in runs:
            rec["ingest_" + key] = {"ms": [round(x, 2) for x in runs[key]], "chunks": outs[key][0],
                                    "unique_chunks": outs[key][1], "stored_bytes": outs[key][2]}
        result["mixes"][name] = rec
        print(json.dumps({name: rec}), flush=True)
        del off, sz_dev
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
