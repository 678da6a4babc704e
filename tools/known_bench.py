"""Ingest against an existing archive (Ingest.run(known=...), hmse_compress_known) on the seed-42 device corpus cut into
files by the size mix of tools/compose_bench.py (log-normal, median 32 KiB, 0 to 8 MiB).

The corpus is ingested once and built into the base archive, which is opened once (archive.Reader, timed).  Snapshots
are the same files with 0, 1, 10, 50 and 100 % of the non-empty files changed by three seeded byte edits each; CDC
resynchronises after an edit, so the share of files changed is not the share of streams copied, which is reported.  One
more snapshot shares next to nothing with its base: the files of the second half of the corpus against a base built from
the first half (the corpus repeats articles, so the halves still share some streams).  For each snapshot:
  - the whole Ingest.run(files=...) with and without known=, host clock to a device synchronise, alternated, medians;
  - HMSE_T_DEFLATE, HMSE_T_PACK and HMSE_T_KNOWN of each run (CUDA events inside the library);
  - the streams copied and compressed, and whether every field of the result equals the plain run;
  - one IngestStream line: the first --stream-gb GB of the snapshot from pinned host memory, with and without known=,
    and HMSE_T_KNOWN per piece (the digest table is rebuilt for every piece, at O(stored chunks of the base)).
Records the GPU name and power limit, writes one JSON (default profiles/known_bench.json) and fails without a GPU.
`python tools/known_bench.py [--gb 10]`."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from compose_bench import gpu_facts, size_mix  # noqa: E402

T_DEFLATE, T_PACK, T_KNOWN = 4, 5, 14
FIELDS = ("cuts", "digests", "canon", "is_first", "select", "blob", "offsets", "file_chunk")


def timers(ctx):
    out = {}
    for name, i in (("deflate", T_DEFLATE), ("pack", T_PACK), ("known", T_KNOWN)):
        f = C.c_float(0)
        out[name] = round(f.value, 3) if ctx.lib.hmse_timing_ms(ctx.h, i, C.byref(f)) == 0 else None
    return out


def med(xs):
    xs = [x for x in xs if x is not None]
    return round(statistics.median(xs), 3) if xs else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=10.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--stream-gb", type=float, default=2.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "known_bench.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("known_bench.py needs a CUDA device")
    import hmse_b200
    from hmse_b200 import archive
    from hmse_b200 import corpus as pc
    ctx = hmse_b200.Context(0)
    lib = ctx.lib
    n = int(a.gb * 1e9) & ~15
    zd = pc.zdict()
    ing = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), ctx.stage(zd))
    d = pc.DeviceCorpus(ctx).generate(n)
    sizes = size_mix(n)
    off = np.concatenate([[0], np.cumsum(sizes)])
    base = archive.build(ing.run(d[:n], files=sizes), zd, ctx=ctx)
    res = dict(gpu_facts(), raw_bytes=n, files=int(sizes.size), base=dict(chunks=base.n_chunks, stored_chunks=base.n_unique,
               store_bytes=int(base.store.size)), snapshots={})
    opens = []
    for _ in range(a.reps):
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        rd = archive.Reader(base, ctx)
        torch.cuda.synchronize()
        opens.append(round((time.perf_counter() - w0) * 1e3, 1))
    res["open_base_ms"] = opens
    print(json.dumps(res), flush=True)
    lib.hmse_timing(ctx.h, 1)

    def compare(snap, files, src, stream_bytes):
        plain_ms, known_ms, tp, tk, equal = [], [], [], [], True
        for r in range(a.reps + 1):   # the first pair warms up and is not recorded
            for kind in (("plain", "known") if r % 2 else ("known", "plain")):
                lib.hmse_timing(ctx.h, 1)
                torch.cuda.synchronize()
                w0 = time.perf_counter()
                out = ing.run(snap, files=files, known=src if kind == "known" else None)
                torch.cuda.synchronize()
                ms = (time.perf_counter() - w0) * 1e3
                if r:
                    (known_ms if kind == "known" else plain_ms).append(ms)
                    (tk if kind == "known" else tp).append(timers(ctx))
                if kind == "plain":
                    plain = out
                else:
                    got = out
            equal = equal and all(torch.equal(getattr(got, f), getattr(plain, f)) for f in FIELDS)
            del out, plain
        line = dict(equal=equal, stats=got.stats, streams=int(got.select.numel()),
                    copied_share=round(got.stats["copied"] / max(1, got.select.numel()), 4),
                    run_plain_ms=[round(x, 1) for x in plain_ms], run_known_ms=[round(x, 1) for x in known_ms],
                    run_plain_ms_median=med(plain_ms), run_known_ms_median=med(known_ms),
                    plain_timers_median={k: med([t[k] for t in tp]) for k in ("deflate", "pack", "known")},
                    known_timers_median={k: med([t[k] for t in tk]) for k in ("deflate", "pack", "known")})
        del got
        # the same snapshot streamed from pinned host memory (no files: one stream), its first stream_bytes
        host = torch.empty(stream_bytes, dtype=torch.uint8, pin_memory=True)
        host.copy_(snap[:stream_bytes])
        st = hmse_b200.IngestStream(ctx, hmse_b200.CDCConfig(), ctx.stage(zd))
        s_plain, s_known, s_equal = [], [], True
        for r in range(a.reps + 1):
            for kind in (("plain", "known") if r % 2 else ("known", "plain")):
                torch.cuda.synchronize()
                w0 = time.perf_counter()
                out = st.run(host, known=src if kind == "known" else None)
                ms = (time.perf_counter() - w0) * 1e3
                if r:
                    (s_known if kind == "known" else s_plain).append(ms)
                if kind == "plain":
                    sp = {f: getattr(out, f).clone() for f in ("cuts", "canon", "offsets", "blob")}
                    continue
                sk = {f: getattr(out, f).clone() for f in ("cuts", "canon", "offsets", "blob")}
                s_stats = out.stats
            s_equal = s_equal and all(torch.equal(sp[f], sk[f]) for f in sp)
        per_piece = []
        st.timing_hook = lambda: per_piece.append(timers(ctx)["known"])
        st.run(host, known=src)
        st.timing_hook = None
        line["stream"] = dict(bytes=stream_bytes, equal=s_equal, stats=s_stats, pieces=len(per_piece),
                              run_plain_ms=[round(x, 1) for x in s_plain], run_known_ms=[round(x, 1) for x in s_known],
                              run_plain_ms_median=med(s_plain), run_known_ms_median=med(s_known),
                              known_ms_per_piece_median=med(per_piece))
        del host, st
        return line

    rng = np.random.default_rng(42)
    nonempty = np.flatnonzero(sizes > 0)
    snap = torch.empty(n + 64, dtype=torch.uint8, device=ctx.tdev)
    sb = int(a.stream_gb * 1e9) & ~15
    for pct in (0, 1, 10, 50, 100):
        snap[:n].copy_(d[:n])
        ch = rng.choice(nonempty, int(round(nonempty.size * pct / 100)), replace=False)
        pos = (off[ch][:, None] + (rng.random((ch.size, 3)) * sizes[ch][:, None]).astype(np.int64)).reshape(-1)
        if pos.size:
            p = torch.from_numpy(pos).to(ctx.tdev)
            snap[p] ^= 0x5A
        line = dict(files_changed_pct=pct, files_changed=int(ch.size), **compare(snap[:n], sizes, rd, min(sb, n)))
        res["snapshots"]["changed_%d_pct" % pct] = line
        print(pct, json.dumps(line), flush=True)
    # next to nothing in common: the second half of the files against a base of the first half
    half = sizes.size // 2
    cut = int(off[half])
    base_a = archive.build(ing.run(d[:cut], files=sizes[:half]), zd, ctx=ctx)
    rd_a = archive.Reader(base_a, ctx)
    snap[:n - cut].copy_(d[cut:n])
    line = dict(base="first half of the files", snapshot="second half", **compare(snap[:n - cut], sizes[half:], rd_a, min(sb, n - cut)))
    res["snapshots"]["disjoint_halves"] = line
    print("disjoint", json.dumps(line), flush=True)
    lib.hmse_timing(ctx.h, 0)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
