"""Composing archives (archive.compose, hmse_compose) on the seed-42 device corpus cut into files by a seeded size mix
(log-normal, median 32 KiB, 0 to 8 MiB) and ingested as two archives, one per half of the files.

Times three composes: the two archives merged, one archive merged with itself, and a subset of half the files (every
other file of both archives).  For each: the device time of hmse_compose (HMSE_T_COMPOSE events), the wall time of the
whole compose() call with its sources already open, the copy of the output to the host (the same bytes copied from the
device on their own), and a device-to-device copy of as many bytes as the output store (events), the floor of the
gather step.  The source opens (archive.Reader) are timed on their own.  Records the GPU name and power limit, writes
one JSON (default profiles/compose_bench.json) and fails without a GPU.  `python tools/compose_bench.py [--gb 10]`."""
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

T_COMPOSE = 13


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


def size_mix(n, seed=42):
    rng = np.random.default_rng(seed)
    sizes = np.clip(rng.lognormal(np.log(32 << 10), 1.5, n // (16 << 10) + 16).astype(np.int64), 0, 8 << 20)
    sizes = sizes[:np.searchsorted(np.cumsum(sizes), n)]
    return np.concatenate([sizes, [n - int(sizes.sum())]])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=10.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "compose_bench.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("compose_bench.py needs a CUDA device")
    import hmse_b200
    from hmse_b200 import archive
    from hmse_b200 import corpus as pc
    ctx = hmse_b200.Context(0)
    lib = ctx.lib
    n = int(a.gb * 1e9) & ~15
    zd = pc.zdict()
    t0 = time.perf_counter()
    d = pc.DeviceCorpus(ctx).generate(n)[:n]
    sizes = size_mix(n)
    half = sizes.size // 2
    cut = int(sizes[:half].sum())
    ars = []
    for lo, hi, sz in ((0, cut, sizes[:half]), (cut, n, sizes[half:])):
        r = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), ctx.stage(zd)).run(ctx.stage(d[lo:hi]), files=sz)
        ars.append(archive.build(r, zd, ctx=ctx))
        del r
    del d
    torch.cuda.synchronize()
    A, B = ars
    res = dict(gpu_facts(), raw_bytes=n, files=int(sizes.size), build_s=round(time.perf_counter() - t0, 1),
               sources=[dict(chunks=x.n_chunks, stored_chunks=x.n_unique, store_bytes=int(x.store.size), files=x.n_files) for x in ars],
               cases={})
    print(json.dumps(res), flush=True)
    opens = []
    for _ in range(a.reps):
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        ra, rb = archive.Reader(A, ctx), archive.Reader(B, ctx)
        torch.cuda.synchronize()
        opens.append((time.perf_counter() - w0) * 1e3)
    res["open_both_ms"] = [round(x, 1) for x in opens]
    lib.hmse_timing(ctx.h, 1)
    cases = {"merge_two": [(ra, None), (rb, None)], "merge_with_itself": [(ra, None), (ra, None)],
             "subset_half_the_files": [(ra, list(range(0, A.n_files, 2))), (rb, list(range(0, B.n_files, 2)))]}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for name, parts in cases.items():
        walls, devs, d2h, floor = [], [], [], []
        st = {}
        for _ in range(a.reps):
            torch.cuda.synchronize()
            w0 = time.perf_counter()
            out = archive.compose(parts, ctx=ctx, stats=st)
            walls.append((time.perf_counter() - w0) * 1e3)
            ms = C.c_float(0)
            ctx.check(lib.hmse_timing_ms(ctx.h, T_COMPOSE, C.byref(ms)))
            devs.append(ms.value)
            nb = int(out.store.size) + out.index.nbytes + out.pointers.nbytes + (out.delta_store.size if out.n_delta else 0)
            src = torch.empty(nb, dtype=torch.uint8, device=ctx.tdev)
            dst = torch.empty(int(out.store.size) + 64, dtype=torch.uint8, device=ctx.tdev)
            torch.cuda.synchronize()
            w0 = time.perf_counter()
            src.cpu()
            d2h.append((time.perf_counter() - w0) * 1e3)
            ev[0].record()
            dst[:out.store.size].copy_(src[:out.store.size])
            ev[1].record()
            torch.cuda.synchronize()
            floor.append(ev[0].elapsed_time(ev[1]))
            del src, dst
        res["cases"][name] = dict(stats=st, out_chunks=out.n_chunks, out_files=out.n_files,
                                  compose_device_ms=[round(x, 2) for x in devs], compose_call_ms=[round(x, 1) for x in walls],
                                  output_d2h_copy_ms=[round(x, 1) for x in d2h], store_d2d_copy_ms=[round(x, 2) for x in floor],
                                  compose_device_ms_median=round(statistics.median(devs), 2),
                                  store_d2d_copy_ms_median=round(statistics.median(floor), 2))
        print(name, json.dumps(res["cases"][name]), flush=True)
    lib.hmse_timing(ctx.h, 0)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
