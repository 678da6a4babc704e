#!/usr/bin/env python
"""bench.py - ingest GB/s of the HMSE data-reduction hot path (CDC + SHA-256 + dedup + DEFLATE).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the CPU oracle on the host cores
    python bench.py ... --dump-outputs DIR                   # also the last timed step's result as DIR/*.npy

One step = one pass of the hot path over one batch of synthetic templated-wiki text (seed 42,
generated on the device): at N = 1 BASELINE.json configs[1] (10 GB on one B200); at N > 1 every
rank owns a 10 GB byte-range shard of ONE N x 10 GB stream (boundary resync + global dedup over an
NCCL all-to-all), i.e. weak scaling.  Prints ONE JSON line (rank 0).  GB = 1e9 bytes.

    --config 4   BASELINE.json configs[3]: ONE 100 GB high-redundancy stream (>= 60 % exact duplicates) split into N
                 byte-range shards (strong scaling, N = 2 / 4 / 8), global dedup by digest prefix
    --config 5   BASELINE.json configs[4]: MinHash (128 perms) + LSH (32 bands) over >= 50 M chunks across N GPUs,
                 generated and consumed shard by shard, band-partitioned all-to-all, bucket sort on the band owners
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ingest GB/s (CDC+SHA-256+dedup+DEFLATE)"
UNIT = "GB/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gb", type=float, default=10.0, help="bytes per GPU per step, in GB (1e9)")
    ap.add_argument("--cpu-sample-mib", type=int, default=128)
    ap.add_argument("--piece-mib", type=int, default=2048, help="piece size of the streaming end-to-end path")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the full-size inflate + digest round-trip check")
    ap.add_argument("--no-l4", action="store_true", help="skip the (untimed into `value`) L4 MinHash/LSH/delta pass")
    ap.add_argument("--config", type=int, default=2, choices=[2, 4, 5], help="BASELINE.json configuration (1-based); 2 is the headline")
    ap.add_argument("--total-gb", type=float, default=100.0, help="--config 4: bytes of the ONE stream, in GB")
    ap.add_argument("--chunks-m", type=float, default=50.0, help="--config 5: millions of chunks over all GPUs")
    ap.add_argument("--batch-gb", type=float, default=10.0, help="--config 5: bytes generated and signed per batch per GPU")
    ap.add_argument("--verify-gib", type=float, default=0.0,
                    help="bytes per rank the CPU oracle re-walks in `verify` (GiB from the shard's entry; 0 = the whole shard)")
    ap.add_argument("--no-oracle", action="store_true", help="skip the CPU-oracle leg of `verify` (cuts, digests, canon)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the result of this project's path (--impl ours)")
    return args


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


DUMP_SEED = 20260   # the rows a dump keeps depend on this seed, the array's length and the number of ranks only


def dump_rows(n, cap):
    """Indices of the rows of an n-row array that a dump keeps: all of them, or a sorted seeded sample of `cap`."""
    import numpy as np
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, cap, replace=False))


def dump_outputs(out_dir, arrays, counts, rank, world):
    """Writes what the timed path returned in its last step, so that two builds run with the same arguments (the same
    seeded input) can be compared output for output: DIR/<name>.npy per array and DIR/counts.npy, with the suffix
    .rank<r> at N > 1.  arrays: name -> (tensor, kind, rows).  kind says how values become float32 / float64 exactly:
    "byte" (uint8 / bool -> float32), "int" (integers below 2^53 -> float64), "u32" (32-bit patterns -> float64), "u64"
    (64-bit patterns -> float64 pairs (high, low 32 bits) in a last axis of 2).  rows: the most rows of the array the
    whole dump keeps, split evenly among the ranks; a rank with more keeps the seeded sample dump_rows(n, rows // N).
    The callers' row limits keep a dump under 64 MB whatever N is."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    sfx = "" if world == 1 else ".rank%d" % rank
    for name, (t, kind, rows) in arrays.items():
        keep = torch.from_numpy(dump_rows(int(t.shape[0]), max(1, rows // world)))
        a = t[keep.to(t.device)].cpu().numpy()
        if kind == "byte":
            a = a.astype(np.float32)
        elif kind == "u32":
            a = a.view(np.uint32).astype(np.float64)
        elif kind == "u64":
            u = a.view(np.uint64)
            a = np.stack([u >> np.uint64(32), u & np.uint64(0xFFFFFFFF)], axis=-1).astype(np.float64)
        else:
            a = a.astype(np.float64)
        np.save(os.path.join(out_dir, name + sfx + ".npy"), a)
    np.save(os.path.join(out_dir, "counts" + sfx + ".npy"), np.array(counts, dtype=np.float64))


def dump_ingest(out_dir, res, rank, world):
    """The IngestResult of --config 2 / 4: cuts, digests [n, 32], canon, is_first, select, offsets, blob and counts =
    [entry, id_base, chunks, streams, blob bytes].  At most 2^17 rows of each per-chunk / per-stream array and 2^20 bytes
    of the blob: 26 MB in all."""
    rows = 1 << 17
    dump_outputs(out_dir, {"cuts": (res.cuts, "int", rows), "digests": (res.digests, "byte", rows),
                           "canon": (res.canon, "int", rows), "is_first": (res.is_first, "byte", rows),
                           "select": (res.select, "int", rows), "offsets": (res.offsets, "int", rows),
                           "blob": (res.blob, "byte", 1 << 20)},
                 [res.entry, res.id_base, res.n_chunks, res.select.numel(), res.blob.numel()], rank, world)


def dump_similarity(out_dir, out, rank, world):
    """One step of --config 5: cuts, sig [n, 128], keys [n, 32] (band keys of this rank's chunks), the sorted triples
    (band, key, id) of the bands this rank owns, and counts = [entry, id_base, chunks of the stream, chunks, triples].
    At most 2^14 rows of cuts / sig / keys and 2^17 triples: 30 MB in all."""
    import torch
    rows, trip = 1 << 14, 1 << 17
    none = torch.empty(0, dtype=torch.int64)
    band, key, ids = (none, none, none) if out["band"] is None else (out["band"], out["key"], out["ids"])
    dump_outputs(out_dir, {"cuts": (out["cuts"], "int", rows), "sig": (out["sig"], "u32", rows),
                           "keys": (out["keys"], "u64", rows), "band": (band, "int", trip), "key": (key, "u64", trip),
                           "ids": (ids, "int", trip)},
                 [out["entry"], out["id_base"], out["n_total"], out["cuts"].numel(), band.numel()], rank, world)


# ------------------------------------------------------------------------------------------------
# CPU oracle legs (the only places that import oracle/)
# ------------------------------------------------------------------------------------------------
def _oracle_pass(data, zd):
    import numpy as np
    import oracle
    cuts = oracle.chunk(data)
    dg = oracle.digest(data, cuts)
    canon, first = oracle.dedup(dg)
    blob, offs = oracle.compress(data, cuts, np.flatnonzero(first), zd)
    return cuts.size, int(first.sum()), blob.size


def cpu_baseline(sample_mib: int):
    """One process, the Python/NumPy + hashlib + zlib oracle on a bounded sample of the workload."""
    from oracle import corpus
    data = corpus.generate(sample_mib << 20)
    zd = corpus.zdict()
    t = time.perf_counter()
    n_chunks, n_first, out = _oracle_pass(data, zd)
    dt = time.perf_counter() - t
    return {"value": data.size / dt / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "first %d MiB of the same seed-42 corpus, oracle.chunk (NumPy) + hashlib + dict dedup + zlib-6 "
                      "with the preset dictionary, %.1f s, %d chunks, %d unique" % (sample_mib, dt, n_chunks, n_first)}


def _ref_worker(conn, slice_mib, idx):
    """One oracle process: owns one slice of the corpus; phase 1 = chunk + digest, phase 2 = compress
    the chunks the parent's global dedup kept."""
    import numpy as np
    import oracle
    from oracle import corpus
    data = corpus.generate(slice_mib << 20, first_article=idx * 997)
    zd = corpus.zdict()
    conn.send("ready")
    cuts = None
    while True:
        msg = conn.recv()
        if msg is None:
            return
        if msg == "p1":
            cuts = oracle.chunk(data)
            conn.send(oracle.digest(data, cuts).tobytes())
        else:
            keep = np.frombuffer(msg, dtype=np.uint8).astype(bool)
            blob, _ = oracle.compress(data, cuts, np.flatnonzero(keep), zd)
            conn.send(blob.size)


def run_reference(args):
    """The oracle on every host core: workers chunk+digest their slice, the parent dedups
    globally, workers compress their first occurrences.  Each step is a bounded sample."""
    import multiprocessing as mp
    import numpy as np
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    procs = max(1, min(os.cpu_count() or 1, 64))
    slice_mib = 16
    ctx = mp.get_context("spawn")
    conns, ps = [], []
    for i in range(procs):
        a, b = ctx.Pipe()
        p = ctx.Process(target=_ref_worker, args=(b, slice_mib, i), daemon=True)
        p.start()
        conns.append(a)
        ps.append(p)
    for c in conns:
        assert c.recv() == "ready"

    def step():
        for c in conns:
            c.send("p1")
        digs = [c.recv() for c in conns]
        alld = np.frombuffer(b"".join(digs), dtype=np.uint8).reshape(-1, 32)
        _, first = oracle.dedup(alld)
        pos = 0
        for c, dbytes in zip(conns, digs):
            k = len(dbytes) // 32
            c.send(first[pos:pos + k].astype(np.uint8).tobytes())
            pos += k
        return sum(c.recv() for c in conns)

    for _ in range(args.warmup):
        step()
    t = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t) / args.steps
    for c in conns:
        c.send(None)
    for p in ps:
        p.join(timeout=10)
    nbytes = procs * (slice_mib << 20)
    val = nbytes / dt / 1e9
    sample = "%d oracle processes (os.cpu_count()=%s) x %d MiB slices of the seed-42 corpus per step" % (
        procs, os.cpu_count(), slice_mib)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "NOT the 10 GB stream of configs[1]: a bounded sample of the same generator and pipeline (CDC + "
                                   "SHA-256 + global dedup + zlib-6 with the preset dictionary) on the CPU oracle - " + sample +
                                   "; the slices start at articles 0, 997, 1994, ... so their duplicate rate differs from the 10 GB "
                                   "stream's",
                       "same_workload_as_gpu_arm": False},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def oracle_shard_check(host, entry, own_end, eof, cuts_gpu, digests_gpu, cfg_dict, limit_bytes):
    """CHECKER, not timed into anything: the CPU oracle (Algorithm 1 in C + hashlib) re-walks this rank's shard from
    its entry over the host copy of the same bytes and must reproduce the GPU's cut list and every digest of the range.
    host: uint8 numpy view of the shard buffer (owned bytes + look-ahead); cuts_gpu / digests_gpu: numpy results of the
    GPU (cuts relative to the buffer).  limit_bytes: 0 = up to own_end, else the first limit_bytes after the entry.
    Returns a dict; `exit` = the last oracle cut when the whole shard was walked (the next shard's entry + own_end)."""
    import numpy as np
    import oracle
    from oracle.config import CDCConfig as OCfg
    cfg = OCfg(**cfg_dict)
    t0 = time.perf_counter()
    lim = own_end if not limit_bytes else min(own_end, entry + int(limit_bytes))
    whole = lim == own_end
    last = whole and eof
    view = host if last else host[:min(host.size, lim + cfg.max_size)]
    want = oracle.chunk_c(view, cfg, entry=entry, n_own=lim, eof=last)
    k = want.size
    cuts_ok = bool(cuts_gpu.size >= k and np.array_equal(cuts_gpu[:k], want) and (not whole or cuts_gpu.size == k))
    t1 = time.perf_counter()
    want_dg = oracle.digest_mt(view, want, start0=entry)
    dg = digests_gpu[:k]
    dg_ok = bool(dg.shape[0] == k and np.array_equal(dg, want_dg))
    xo = np.bitwise_xor.reduce(want_dg.view(np.uint64), axis=0) if k else np.zeros(4, dtype=np.uint64)
    t2 = time.perf_counter()
    return {"cuts_equal": cuts_ok, "digests_equal": dg_ok, "chunks": int(k), "bytes": int(lim - entry), "whole_shard": whole,
            "exit": int(want[-1]) if k else int(entry), "xor": "".join("%016x" % int(v) for v in xo),
            "chunk_s": t1 - t0, "digest_s": t2 - t1}


def zlib_sample_check(host, entry, cuts_np, sel_np, blob_dev, offs_dev, zdict_bytes, n_sample, seed=7):
    """CHECKER: n_sample of the compressed streams go through STOCK zlib (with the preset dictionary) on the host and
    must inflate to the chunk's bytes; the GPU read path (`verify.inflate_failed`) covers all of them."""
    import zlib
    import numpy as np
    import torch
    m = int(sel_np.size)
    if m == 0:
        return 0, 0
    rng = np.random.default_rng(seed)
    pick = np.sort(rng.choice(m, min(m, n_sample), replace=False))
    offs = offs_dev.cpu().numpy()
    starts = np.concatenate([[entry], cuts_np[:-1]]).astype(np.int64)
    bad = 0
    for k in pick.tolist():
        stream = blob_dev[int(offs[k]):int(offs[k + 1])].cpu().numpy().tobytes()
        j = int(sel_np[k])
        try:
            do = zlib.decompressobj(zdict=zdict_bytes) if zdict_bytes else zlib.decompressobj()
            raw = do.decompress(stream) + do.flush()
            bad += raw != host[starts[j]:int(cuts_np[j])].tobytes()
        except zlib.error:
            bad += 1
    return int(pick.size), int(bad)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import ctypes as C
    import torch
    import hmse_b200
    from hmse_b200 import corpus as pcorpus

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: hmse_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    # pinned host buffers should live on the GPU's own NUMA node (matters for the end-to-end leg at N > 1)
    numa = hmse_b200.sharding.bind_to_gpu_numa(local) if os.environ.get("HMSE_NO_NUMA_BIND") is None else None
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = hmse_b200.Context(local)
    lib = ctx.lib
    dev = ctx.tdev
    cfg = hmse_b200.CDCConfig()
    shard = int(args.gb * 1e9)
    shard -= shard % 16
    total = shard * world
    eof = rank == world - 1
    n_avail = shard if eof else shard + cfg.max_size
    gen = pcorpus.DeviceCorpus(ctx)
    d = gen.generate(n_avail, byte_off=rank * shard)
    zd = ctx.stage(pcorpus.zdict())
    torch.cuda.synchronize()

    if world > 1:
        pipe = hmse_b200.ShardedIngest(ctx, cfg, zd)
        run = lambda buf: pipe.run(buf, shard, eof)  # noqa: E731
    else:
        pipe = hmse_b200.Ingest(ctx, cfg, zd)
        run = lambda buf: pipe.run(buf)  # noqa: E731

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- device-resident throughput -------------------------------------------------------------
    res = None
    for _ in range(args.warmup):
        res = run(d)
    lib.hmse_timing(ctx.h, 1)
    stage_names = ["scan", "resolve", "sha256", "dedup", "deflate", "pack"]
    stage_ms = {k: 0.0 for k in stage_names}
    parse = {"ms": 0.0, "timed": 0, "launches": 0, "token_bytes": 0, "in_bytes": 0, "chunks": 0}
    xch, xch_ms = None, 0.0
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = lib.hmse_launch_count(ctx.h)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = run(d)
        f = C.c_float(0)
        for i, k in enumerate(stage_names):   # event reads only; the stream is already drained by the API
            if lib.hmse_timing_ms(ctx.h, i, C.byref(f)) == 0:
                stage_ms[k] += f.value
        st4 = (C.c_uint64 * 4)()
        pn = C.c_uint32(0)
        if lib.hmse_compress_stats(ctx.h, st4, C.byref(f), C.byref(pn)) == 0 and pn.value:
            parse["ms"] += f.value
            parse["timed"] += pn.value
            parse["launches"] += st4[0]
            parse["token_bytes"] += 2 * st4[1]
            parse["in_bytes"] += st4[2]
            parse["chunks"] += st4[3]
        if world > 1:
            xch = ctx.exchange_stats()     # the dedup exchange (the last NCCL region of a step)
            xch_ms += xch["ms"] or 0.0
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    launches = (lib.hmse_launch_count(ctx.h) - launches0) // max(1, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    stage_ms = {k: v / args.steps for k, v in stage_ms.items()}
    value = total / (ms * 1e-3) / 1e9
    if args.dump_outputs:
        dump_ingest(args.dump_outputs, res, rank, world)

    # ---- pipeline facts for the roofline ---------------------------------------------------------
    n_chunks = res.n_chunks
    cuts = res.cuts
    starts = torch.cat([torch.full((1,), res.entry, dtype=torch.int64, device=dev), cuts[:-1]])
    lens = cuts - starts
    sel_bytes = int(lens[res.select].sum()) if res.select.numel() else 0
    out_bytes = int(res.blob.numel())
    peak, peak_src = measured_peak()
    # Dominant kernel: parse_kernel (>= 60 % of the device time, profiles/).  Per launch (one batch of <= 32768
    # chunks): algorithmic bytes = chunk bytes read once + 16-bit token words + 1312 B of symbol counts and record per
    # chunk (DESIGN.md section 4), divided by the average launch span measured with one CUDA-event pair per launch.
    n_l = max(1, parse["launches"])
    alg_per_launch = (parse["in_bytes"] + parse["token_bytes"] + 1312 * parse["chunks"]) / n_l
    ms_per_launch = parse["ms"] / max(1, parse["timed"])
    parse_gbs = alg_per_launch / (ms_per_launch * 1e-3) / 1e9 if ms_per_launch > 0 else 0.0
    defl_bytes = sel_bytes + out_bytes
    defl_gbs = defl_bytes / (stage_ms["deflate"] * 1e-3) / 1e9 if stage_ms["deflate"] > 0 else 0.0
    traffic = traffic_note = ncu_facts = None
    try:
        with open(os.path.join(ROOT, "profiles", "deflate_traffic.json")) as f:
            tj = json.load(f)
            traffic = tj.get("dram_bytes_per_launch")
            traffic_note = tj.get("note")
            ncu_facts = tj.get("ncu")
    except Exception:  # noqa: BLE001
        pass
    # The kernel is bound by instruction issue, not by HBM (ncu: DRAM ~1 % of peak).  Its issue-rate fraction: warp
    # instructions per launch = (ncu-counted warp instructions per input byte of the committed capture) x (input bytes
    # of the live launch), over the live launch time, against 4 schedulers x 1 warp instruction per cycle per SM.
    issue = None
    sm_clock_hz = 1965e6
    try:
        props = torch.cuda.get_device_properties(local)
        n_sm = props.multi_processor_count
        if ncu_facts and ncu_facts.get("warp_instructions") and ncu_facts.get("input_bytes") and ms_per_launch > 0:
            wi_per_byte = ncu_facts["warp_instructions"] / ncu_facts["input_bytes"]
            in_per_launch = parse["in_bytes"] / n_l
            ach = wi_per_byte * in_per_launch / (ms_per_launch * 1e-3)
            pk = n_sm * 4 * sm_clock_hz
            issue = {"warp_instr_per_input_byte": wi_per_byte, "achieved_warp_instr_per_s": ach, "peak_warp_instr_per_s": pk,
                     "frac": ach / pk, "peak_source": "%d SMs x 4 schedulers x 1965 MHz (MEASURED_PEAKS.json sm_max_mhz)" % n_sm,
                     "ncu_issue_active_pct": ncu_facts.get("issue_active_pct")}
    except Exception:  # noqa: BLE001
        issue = None
    roofline = {"bound": "issue", "kernel": "parse_kernel (match search + parse of one batch of chunks; the other kernels of "
                                            "the stage are listed under other_kernels)",
                "frac_issue": issue["frac"] if issue else None, "issue": issue,
                "achieved": parse_gbs, "peak": peak, "unit": "GB/s", "frac": parse_gbs / peak, "traffic": traffic,
                "traffic_note": traffic_note, "ncu": ncu_facts, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_per_launch, "ms_per_launch": ms_per_launch,
                "launches_per_step": parse["launches"] / max(1, args.steps), "launches_timed": parse["timed"],
                "other_kernels": {k: {"ms": stage_ms[k],
                                      "GB/s": (shard / (stage_ms[k] * 1e-3) / 1e9) if stage_ms[k] > 0 else None}
                                  for k in ("scan", "resolve", "sha256")},
                "deflate_stage": {"ms": stage_ms["deflate"], "algorithmic_bytes": defl_bytes, "GB/s": defl_gbs,
                                  "frac": defl_gbs / peak},
                "pipeline_frac": ((total + sum_over_ranks(out_bytes) + 40 * sum_over_ranks(n_chunks)) / (ms * 1e-3) / 1e9)
                / (peak * world)}

    # ---- full-size parity property (not timed into `value`): every compressed stream of the last step goes
    #      through the device read path (hmse_inflate) and the SHA-256 of what comes out must equal the digest
    #      taken from the source chunk - an encode -> decode round trip plus a checksum of checksums ----
    verify = None
    host_in = None
    if not args.no_e2e or (not args.no_verify and not args.no_oracle):
        host_in = torch.empty(n_avail, dtype=torch.uint8, pin_memory=True)   # the end-to-end leg's input; the oracle's too
        host_in.copy_(d)
    if not args.no_verify:
        torch.cuda.synchronize()
        v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        v0.record()
        bad, same = hmse_b200.verify_roundtrip(ctx, res, zd)
        v1.record()
        torch.cuda.synchronize()
        f = C.c_float(0)
        inf_ms = f.value if lib.hmse_timing_ms(ctx.h, 8, C.byref(f)) == 0 else None
        verify = {"streams": int(sum_over_ranks(int(res.select.numel()))), "inflate_failed": int(sum_over_ranks(bad)),
                  "digests_equal": bool(sum_over_ranks(0 if same else 1) == 0),
                  "inflate_ms": inf_ms, "inflate_GBps_out": (sel_bytes / (inf_ms * 1e-3) / 1e9) if inf_ms else None,
                  "total_ms": v0.elapsed_time(v1),
                  "what": "hmse_inflate of every stream + SHA-256 of the output == digest of the source chunk, at full size"}
        if not args.no_oracle:
            # ---- the CPU oracle over the SAME bytes (host copy of this rank's shard buffer): every rank re-walks its
            #      shard from its entry (Algorithm 1 in C), hashes every chunk (hashlib) and compares cut list and digests;
            #      the shard edges chain (entry of rank r == exit of rank r-1, both oracle-checked), so the N cut lists
            #      together equal the single-stream oracle cut list by induction from rank 0's entry 0; the global
            #      canon is checked against the oracle's dedup over the gathered digests ----
            import dataclasses
            import numpy as np
            t_or = time.perf_counter()
            host_np = host_in.numpy()
            cuts_np = res.cuts.cpu().numpy().view(np.uint64)
            dg_np = res.digests.cpu().numpy()
            own_end = n_avail if eof else shard
            oc = oracle_shard_check(host_np, int(res.entry), own_end, eof, cuts_np, dg_np, dataclasses.asdict(cfg),
                                    int(args.verify_gib * (1 << 30)))
            sel_np = res.select.cpu().numpy()
            n_z, bad_z = zlib_sample_check(host_np, int(res.entry), cuts_np, sel_np, res.blob, res.offsets, pcorpus.zdict(), 2000)
            edges_ok, edges = True, 0
            canon_ok = True
            if dist is None:
                import oracle
                wc, _ = oracle.dedup_fast(dg_np)
                canon_ok = bool(np.array_equal(res.canon.cpu().numpy(), wc))
            else:
                # (entry, oracle exit, own_end, n chunks) of every rank
                mine = torch.tensor([int(res.entry), oc["exit"], own_end, n_chunks, int(res.id_base)], dtype=torch.int64, device=dev)
                allv = [torch.empty_like(mine) for _ in range(world)]
                dist.all_gather(allv, mine)
                allv = [t.tolist() for t in allv]
                for r in range(1, world):
                    edges += 1
                    edges_ok = edges_ok and oc["whole_shard"] and allv[r][0] == allv[r - 1][1] - allv[r - 1][2]
                    edges_ok = edges_ok and allv[r][4] == allv[r - 1][4] + allv[r - 1][3]
                # global dedup: digests gathered on rank 0 (padded), oracle dedup there, expected canon broadcast back
                nmax = max(v[3] for v in allv)
                pad = torch.zeros(nmax, 32, dtype=torch.uint8, device=dev)
                pad[:n_chunks] = res.digests
                gl = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
                dist.gather(pad, gl, dst=0)
                n_tot = sum(v[3] for v in allv)
                want_canon = torch.empty(n_tot, dtype=torch.int64, device=dev)
                if rank == 0:
                    import oracle
                    alld = np.concatenate([g[:allv[r][3]].cpu().numpy() for r, g in enumerate(gl)])
                    wc, _ = oracle.dedup_fast(alld)
                    want_canon.copy_(torch.from_numpy(wc))
                    del gl, alld
                dist.broadcast(want_canon, src=0)
                base_id = int(res.id_base)
                canon_ok = bool(torch.equal(want_canon[base_id:base_id + n_chunks], res.canon))
                del want_canon, pad
            all_ok = oc["cuts_equal"] and oc["digests_equal"] and canon_ok and bad_z == 0
            verify.update({
                "oracle_equal": bool(sum_over_ranks(0 if all_ok else 1) == 0) and edges_ok,
                "edges_checked": edges, "edges_equal": edges_ok,
                "oracle": {"what": "per rank: oracle.chunk_c (FastCDC Algorithm 1 in C) from the shard's entry + hashlib SHA-256 of every "
                                   "chunk over the host copy of the same bytes == GPU cuts and digests; entry of rank r == oracle "
                                   "exit of rank r-1; oracle dedup over all gathered digests == GPU canon; a sample of streams "
                                   "through stock zlib with the preset dictionary",
                           "cuts_equal": bool(sum_over_ranks(0 if oc["cuts_equal"] else 1) == 0),
                           "digests_equal": bool(sum_over_ranks(0 if oc["digests_equal"] else 1) == 0),
                           "canon_equal": bool(sum_over_ranks(0 if canon_ok else 1) == 0),
                           "chunks_checked": int(sum_over_ranks(oc["chunks"])), "bytes_checked": int(sum_over_ranks(oc["bytes"])),
                           "whole_shards": bool(sum_over_ranks(0 if oc["whole_shard"] else 1) == 0),
                           "zlib_streams_sampled": int(sum_over_ranks(n_z)), "zlib_streams_failed": int(sum_over_ranks(bad_z)),
                           "rank0_digest_xor": oc["xor"], "rank0_chunk_s": oc["chunk_s"], "rank0_digest_s": oc["digest_s"],
                           "host_threads": min(32, os.cpu_count() or 1), "total_s": time.perf_counter() - t_or}})
            del host_np, cuts_np, dg_np

    # ---- L4 similarity layer on the same batch (reported beside the headline metric, not part of it): MinHash ->
    #      band keys -> buckets -> base selection -> delta coding with the 20 % rule, then the read path: every kept
    #      delta is applied to its base on the device and the SHA-256 of the result must equal the chunk's digest ----
    l4 = None
    if not args.no_l4 and world > 1:
        # N > 1: ONE LSH index over the whole stream (ShardedIngest.similarity_delta_global): band keys to the band owners,
        # heads back, roots gathered, bases that live on another GPU fetched over NCCL, then the delta coding; verified by
        # applying every kept delta to its base (local chunk or fetched bytes) and comparing SHA-256 with the chunk's digest
        sim = hmse_b200.SimConfig()
        first_u8 = res.is_first.view(torch.uint8).contiguous()
        g = None
        for l4_pass in range(2):
            g = None
            torch.cuda.synchronize()
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            g = pipe.similarity_delta_global(d, cuts, first_u8, int(res.entry), int(res.id_base), sim, 4)
            g1.record()
            torch.cuda.synchronize()
        l4_ms = max_over_ranks(g0.elapsed_time(g1))
        kept = torch.nonzero(g["base_gid"] >= 0).view(-1)
        same_l4, dbad = True, 0
        if kept.numel():
            bl_ = g["base_loc"][kept]
            is_ext = bl_ >= n_chunks
            both = torch.cat([d, g["ext_data"]])
            e_ = (bl_ - n_chunks).clamp(min=0)
            eo_ = torch.cat([g["ext_off"], g["ext_off"][-1:]])    # (torch.where evaluates both sides: keep e_ + 1 in range)
            bo = torch.where(is_ext, d.numel() + eo_[e_], starts[bl_.clamp(max=n_chunks - 1)]).contiguous()
            bl = torch.where(is_ext, eo_[e_ + 1] - eo_[e_], lens[bl_.clamp(max=n_chunks - 1)]).to(torch.int32).contiguous()
            out_off = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(lens[kept], 0)])
            doff_k = torch.cat([g["delta_offsets"][kept], g["delta_offsets"][-1:]])
            rebuilt, dstatus, dbad = ctx.delta_apply(g["delta_blob"], doff_k, both, bo, bl, out_off)
            same_l4 = bool(torch.equal(ctx.digest(rebuilt, out_off[1:].contiguous()), res.digests[kept])) and dbad == 0
            del both, rebuilt
        in_store = (g["base_gid"][res.select] >= 0)
        clen = res.offsets[1:] - res.offsets[:-1]
        kept_deflated = int(clen[in_store].sum())
        n_cross = int((g["base_loc"][kept] >= n_chunks).sum()) if kept.numel() else 0
        l4 = {"what": "GLOBAL L4 over the %d x %.0f GB stream: MinHash of the first occurrences on their own rank, band keys to the band "
                      "owners (hmse_lsh_exchange), bucket heads back (hmse_alltoallv), roots gathered, remote base chunks fetched, delta "
                      "coding with the 20 %% rule; second of two passes, whole layer timed with CUDA events, max over ranks" % (world, args.gb),
              "ms": l4_ms, "GB/s": total / (l4_ms * 1e-3) / 1e9,
              "deltas_kept": int(sum_over_ranks(int(kept.numel()))), "deltas_with_base_on_another_gpu": int(sum_over_ranks(n_cross)),
              "remote_bases_fetched": int(sum_over_ranks(g["n_remote"])), "remote_base_bytes": int(sum_over_ranks(int(g["ext_off"][-1]))),
              "kept_raw_bytes": int(sum_over_ranks(int(lens[kept].sum()) if kept.numel() else 0)),
              "delta_bytes": int(sum_over_ranks(int(g["delta_blob"].numel()))),
              "same_chunks_deflated_bytes": int(sum_over_ranks(kept_deflated)),
              "store_bytes_saved": int(sum_over_ranks(kept_deflated - int(g["delta_blob"].numel()) - 8 * int(kept.numel()))),
              "read_path": {"deltas_applied": int(sum_over_ranks(int(kept.numel()))), "failed": int(sum_over_ranks(int(dbad))),
                            "digests_equal": bool(sum_over_ranks(0 if same_l4 else 1) == 0)}}
        del g
    elif not args.no_l4:
        sim = hmse_b200.SimConfig()
        usel = res.select                     # first occurrences: the only chunks that are hashed (README.md:1553-1556)
        ones = torch.ones(usel.numel(), dtype=torch.uint8, device=dev)
        for l4_pass in range(2):              # the first pass sizes the scratch buffers (device-synchronising allocations)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(10)]
            torch.cuda.synchronize()
            ev[0].record()
            sig = ctx.minhash(d, cuts, sim, start0=int(res.entry), select=usel)
            ev[1].record()
            keys = ctx.lsh_keys(sig, sim)
            band, key, ids = ctx.lsh_buckets(keys)
            ev[2].record()
            base_u = ctx.delta_bases(band, key, ids, usel.numel(), sim.bands, ones, 4)
            ev[3].record()
            base = torch.full((n_chunks,), -1, dtype=torch.int64, device=dev)   # compacted indices back to chunk indices
            base[usel] = torch.where(base_u >= 0, usel[base_u.clamp(min=0)], base_u)
            n_cand = int((base >= 0).sum())
            ev[4].record()
            dblob, doffs = ctx.delta_encode(d, cuts, base, start0=int(res.entry))
            ev[5].record()
            kept = torch.nonzero(base >= 0).view(-1)
            bj = base[kept]
            out_off = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(lens[kept], 0)])
            doff_k = torch.cat([doffs[kept], doffs[-1:]])
            bo, bl = starts[bj].contiguous(), lens[bj].to(torch.int32).contiguous()
            ev[6].record()
            rebuilt, dstatus, dbad = ctx.delta_apply(dblob, doff_k, d, bo, bl, out_off)
            ev[7].record()
            torch.cuda.synchronize()
            tms = [ev[a_].elapsed_time(ev[b_]) for a_, b_ in ((0, 1), (1, 2), (2, 3), (4, 5), (6, 7))]
        dg2 = ctx.digest(rebuilt, out_off[1:].contiguous()) if kept.numel() else res.digests[:0]
        same_l4 = bool(torch.equal(dg2, res.digests[kept])) and dbad == 0
        kept_raw = int(lens[kept].sum())
        # what the same chunks cost in the chunk store (their zlib streams of this step)
        in_store = (base[res.select] >= 0)
        clen = res.offsets[1:] - res.offsets[:-1]
        kept_deflated = int(clen[in_store].sum())
        l4_ms = sum(tms[:4])
        l4_ms = max_over_ranks(l4_ms)
        l4 = {"what": "MinHash (128 perms, seeds 1..128) + LSH (32 bands x 4 rows) + base selection (min 4 votes, roots only) + "
                      "delta coding (20 %% rule) over the first occurrences of the same %.0f GB batch per GPU, second of two passes, CUDA "
                      "events per stage%s" % (args.gb, "" if world == 1 else "; N > 1: shard-local bases among the chunks that are first in "
                                              "the WHOLE stream (global dedup first), stage times of rank 0, counts summed, GB/s = all shards / slowest rank"),
              "minhash_ms": tms[0], "lsh_keys_buckets_ms": tms[1], "bases_ms": tms[2], "delta_encode_ms": tms[3],
              "delta_apply_ms": tms[4], "GB/s": total / (l4_ms * 1e-3) / 1e9, "minhash_GB/s": sel_bytes / (tms[0] * 1e-3) / 1e9, "minhash_bytes": sel_bytes,
              "candidates": int(sum_over_ranks(n_cand)), "deltas_kept": int(sum_over_ranks(int(kept.numel()))),
              "kept_raw_bytes": int(sum_over_ranks(kept_raw)),
              "delta_bytes": int(sum_over_ranks(int(dblob.numel()))), "same_chunks_deflated_bytes": int(sum_over_ranks(kept_deflated)),
              "store_bytes_saved": int(sum_over_ranks(kept_deflated - int(dblob.numel()) - 8 * int(kept.numel()))),
              "read_path": {"deltas_applied": int(sum_over_ranks(int(kept.numel()))), "failed": int(sum_over_ranks(int(dbad))),
                            "digests_equal": bool(sum_over_ranks(0 if same_l4 else 1) == 0)}}
        del sig, keys, band, key, ids, base, base_u, dblob, doffs, rebuilt

    uniq_chunks = sum_over_ranks(int(res.select.numel()))
    tot_chunks = sum_over_ranks(n_chunks)
    sel_b = sum_over_ranks(sel_bytes)
    out_b = sum_over_ranks(out_bytes)

    lib.hmse_timing(ctx.h, 0)
    # ---- end to end: pinned host input -> device -> results back on the host, every step ----------
    e2e = None
    if not args.no_e2e:
        d2h = 0
        if world == 1:
            # one GPU: the streaming front end - pieces copied in while the previous piece is processed and
            # the one before travels back (hmse_b200.IngestStream); results equal Ingest.run (tests/test_gpu_stream.py)
            del d, res, cuts, starts, lens
            torch.cuda.empty_cache()
            stream_pipe = hmse_b200.IngestStream(ctx, cfg, zd, piece_bytes=args.piece_mib << 20)
            api = ("hmse_b200.IngestStream.run_many(pinned host buffers, one per step): %d MiB pieces, host->device copy of "
                   "piece k+1, pipeline on piece k and device->host copy of the results of piece k-1 (cuts, digests, canon, "
                   "offsets, compressed blob) overlap on three CUDA streams; the next step's input is copied in behind the "
                   "current step's (two device input buffers)" % args.piece_mib)

            step_trace = []

            def e2e_steps(k):
                nonlocal d2h, step_trace
                stream_pipe.trace = []
                for r in stream_pipe.run_many([host_in] * k, host_blob_cap=n_avail // 2 + (1 << 20)):
                    d2h = r.d2h_bytes
                    step_trace = [(lab, round(ms_, 1)) for lab, ms_ in stream_pipe.trace]   # host ms since this step's run() began
                    stream_pipe.trace = []
                stream_pipe.trace = None
        else:
            host_out = pipe.host_buffers(n_avail)
            api = ("hmse_b200.ShardedIngest.run_batches(pinned host shard buffers, host=pinned result buffers): every step's "
                   "input is copied host->device (double-buffered: the copy of step k+1 runs beside the pipeline of step k), "
                   "cuts, digests, canon, offsets and the compressed blob land in pinned host memory each step, the blob "
                   "leaving in 8 pieces while the remaining chunks are compressed")

            def e2e_steps(k):
                nonlocal d2h
                for r in pipe.run_batches([host_in] * k, shard, eof, host=host_out):
                    d2h = r.d2h_bytes

        # as many end-to-end steps as device-resident ones: the first batch's copy-in cannot hide behind a previous step
        # (pipeline fill, ~180 ms at 10 GB), so a region of three steps would charge 60 ms of it to every step
        k_e2e = max(1, args.steps)
        e2e_steps(1)
        barrier()
        if world > 1:
            pipe.trace = []
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        e2e_steps(k_e2e)
        a1.record()
        barrier()
        timeline = step_trace if world == 1 else None
        if world > 1 and pipe.trace:
            # rank 0, per batch, ms since the timed region began: copy-in start / end, pipeline start, all results on the host
            timeline = [[round(a0.elapsed_time(ev), 1) for ev in tup] for tup in pipe.trace]
            pipe.trace = None
        ems = max_over_ranks(a0.elapsed_time(a1)) / k_e2e
        # ---- the host's ceiling for this byte mix: the same host->device and device->host bytes per step, copies only
        #      (no kernels), both directions at once, all ranks at once ----
        cur = torch.cuda.current_stream(local)
        s_up, s_dn = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        c_in = torch.empty(n_avail, dtype=torch.uint8, device=dev)
        c_out = torch.empty(max(d2h, 1), dtype=torch.uint8, device=dev)
        h_out = (stream_pipe._host["blob"] if world == 1 else host_out["blob"])
        if h_out.numel() < d2h:
            h_out = torch.empty(d2h, dtype=torch.uint8, pin_memory=True)

        def copy_steps(k):
            s_up.wait_stream(cur)
            s_dn.wait_stream(cur)
            for _ in range(k):
                with torch.cuda.stream(s_up):
                    c_in.copy_(host_in, non_blocking=True)
                with torch.cuda.stream(s_dn):
                    h_out[:d2h].copy_(c_out[:d2h], non_blocking=True)
            cur.wait_stream(s_up)
            cur.wait_stream(s_dn)

        copy_steps(1)
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        copy_steps(k_e2e)
        c1.record()
        barrier()
        cms = max_over_ranks(c0.elapsed_time(c1)) / k_e2e
        del c_in, c_out
        e2e = {"value": total / (ems * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(sum_over_ranks(n_avail)),
               "d2h_bytes_per_step": int(sum_over_ranks(d2h)), "ms_per_step": ems, "steps": k_e2e, "api": api,
               "host_ceiling_GBps": total / (cms * 1e-3) / 1e9, "host_ceiling_ms_per_step": cms,
               "timeline_rank0_ms": timeline,
               "frac_of_host_ceiling": cms / ems,
               "host_ceiling_what": "the same pinned buffers and bytes per step copied host->device and device->host on two "
                                    "streams with no kernels, all ranks at once, max over ranks"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline(args.cpu_sample_mib)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
                "data": "synthetic",
                "config": {"workload": "BASELINE.json configs[1]: %.0f GB per GPU of seed-42 templated-wiki text generated on "
                                       "the device, FastCDC avg 8 KiB (min 2 KiB, max 32 KiB) + SHA-256 + exact dedup + zlib-"
                                       "format DEFLATE of first occurrences with a 30 KiB preset dictionary" % args.gb,
                           "bytes_per_gpu": shard, "parallelism": "1 GPU" if world == 1 else
                           "byte-range shards of one %d x %.0f GB stream, boundary resync + global dedup by NCCL all-to-all"
                           % (world, args.gb),
                           "l2": "inputs (%.0f GB per step) far exceed the 126 MB L2; no explicit flush" % args.gb,
                           "chunks": int(tot_chunks), "unique_chunks": int(uniq_chunks),
                           "unique_bytes": int(sel_b), "compressed_bytes": int(out_b),
                           "compression_ratio_unique": (sel_b / out_b) if out_b else None},
                "stages_ms": stage_ms,
                "exchange": None if xch is None else {"what": "hmse_dedup_global on rank 0, last step: {digest, gid} records to their owners "
                                                              "(le32(digest) % N) and the answers back, ncclSend/ncclRecv groups inside the library",
                                                      "bytes_sent_rank0": xch["bytes_sent"], "bytes_received_rank0": xch["bytes_received"],
                                                      "records_owned_rank0": xch["owned"], "nccl_ms_rank0": xch_ms / args.steps,
                                                      "resync_rounds": xch["rounds"], "transport": getattr(pipe, "transport", None)},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "verify": verify, "l4": l4, "numa_bind": numa, "gpu_launches": int(launches),
                "clocks": clocks}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def _setup():
    """Process / device / communicator setup shared by the GPU arms."""
    import torch
    import hmse_b200
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: hmse_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = hmse_b200.Context(local)
    dev = ctx.tdev

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def red(x: float, op: str) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
        return float(t.item())

    return world, rank, local, dist, ctx, dev, barrier, red


def _mem_available_gb() -> float:
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) / 1e6
    except Exception:  # noqa: BLE001
        pass
    return 0.0


def run_config4(args):
    """BASELINE.json configs[3]: ONE high-redundancy stream (>= 60 % exact duplicates, README.md:2073; generator knobs
    README.md:2121-2127) of --total-gb GB split into N contiguous byte-range shards - strong scaling - with boundary
    resync and global dedup by digest prefix (hmse_chunk_sharded / hmse_dedup_global, NCCL send/recv over NVLink)."""
    import ctypes as C
    import dataclasses
    import numpy as np
    import torch
    import hmse_b200
    from hmse_b200 import corpus as pcorpus
    world, rank, local, dist, ctx, dev, barrier, red = _setup()
    lib = ctx.lib
    cfg = hmse_b200.CDCConfig()
    total = int(args.total_gb * 1e9)
    shard = (total // world) & ~15
    eof = rank == world - 1
    lo = rank * shard
    n_avail = (total - lo) if eof else shard + cfg.max_size
    ccfg = pcorpus.CorpusConfig.high_redundancy()
    gen = pcorpus.DeviceCorpus(ctx, ccfg)
    d = gen.generate(n_avail, byte_off=lo)
    zd = ctx.stage(pcorpus.zdict())
    torch.cuda.synchronize()
    if world > 1:
        pipe = hmse_b200.ShardedIngest(ctx, cfg, zd)
        run = lambda buf: pipe.run(buf, shard, eof)  # noqa: E731
    else:
        pipe = hmse_b200.Ingest(ctx, cfg, zd)
        run = lambda buf: pipe.run(buf)  # noqa: E731
    res = None
    for _ in range(args.warmup):
        res = None            # (a shard's blob is tens of GB: drop the previous step's before the next is allocated)
        res = run(d)
    lib.hmse_timing(ctx.h, 1)
    names = ["scan", "resolve", "sha256", "dedup", "deflate", "pack"]
    stage_ms = {k: 0.0 for k in names}
    xch_ms, xch = 0.0, None
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    l0 = lib.hmse_launch_count(ctx.h)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = None
        res = run(d)
        f = C.c_float(0)
        for i, k in enumerate(names):
            if lib.hmse_timing_ms(ctx.h, i, C.byref(f)) == 0:
                stage_ms[k] += f.value
        if world > 1:
            xch = ctx.exchange_stats()     # the dedup exchange is the last one of a step
            xch_ms += xch["ms"] or 0.0
    e1.record()
    barrier()
    ms = red(e0.elapsed_time(e1), "max") / args.steps
    launches = (lib.hmse_launch_count(ctx.h) - l0) // max(1, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    lib.hmse_timing(ctx.h, 0)
    stage_ms = {k: v / args.steps for k, v in stage_ms.items()}
    if args.dump_outputs:
        dump_ingest(args.dump_outputs, res, rank, world)
    n_chunks = res.n_chunks
    starts = torch.cat([torch.full((1,), int(res.entry), dtype=torch.int64, device=dev), res.cuts[:-1]])
    lens = res.cuts - starts
    sel_bytes = int(lens[res.select].sum()) if res.select.numel() else 0
    tot_chunks, uniq_chunks = red(n_chunks, "sum"), red(int(res.select.numel()), "sum")
    uniq_bytes, out_bytes = red(sel_bytes, "sum"), red(int(res.blob.numel()), "sum")
    # ---- verification: device read path over everything; CPU oracle over the first --verify-gib of every shard (default
    #      1 GiB here: the shards are 12.5-50 GB) and over the last 64 MiB before every shard edge; global canon against the
    #      oracle's dedup over all gathered digests ----
    verify = None
    if not args.no_verify:
        bad, same = hmse_b200.verify_roundtrip(ctx, res, zd)
        verify = {"streams": int(uniq_chunks), "inflate_failed": int(red(bad, "sum")), "digests_equal": bool(red(0 if same else 1, "sum") == 0)}
        if not args.no_oracle:
            t_or = time.perf_counter()
            lim = int((args.verify_gib or 1.0) * (1 << 30))
            own_end = n_avail if eof else shard
            cuts_np = res.cuts.cpu().numpy().view(np.uint64)
            dg_np = res.digests.cpu().numpy()
            entry = int(res.entry)
            cfgd = dataclasses.asdict(cfg)
            head_n = min(n_avail, entry + lim + cfg.max_size + 64)
            oc = oracle_shard_check(d[:head_n].cpu().numpy(), entry, own_end, eof, cuts_np, dg_np, cfgd, lim)
            # the tail: from the GPU cut nearest below own_end - 64 MiB through the exit (the next shard's entry)
            tail_ok, tail_exit = True, oc["exit"]
            if not oc["whole_shard"]:
                k0 = int(np.searchsorted(cuts_np, np.uint64(max(entry, own_end - (64 << 20)))))
                t_entry = int(cuts_np[k0])
                t_lo = t_entry & ~15
                tail = d[t_lo:].cpu().numpy()
                ot = oracle_shard_check(tail, t_entry - t_lo, own_end - t_lo, eof, cuts_np[k0 + 1:] - np.uint64(t_lo), dg_np[k0 + 1:], cfgd, 0)
                tail_ok = ot["cuts_equal"] and ot["digests_equal"]
                tail_exit = ot["exit"] + t_lo
                oc["chunks"] += ot["chunks"]
                oc["bytes"] += ot["bytes"]
                del tail
            edges_ok, edges, canon_ok = True, 0, True
            if dist is None:
                import oracle
                wc, _ = oracle.dedup_fast(dg_np)
                canon_ok = bool(np.array_equal(res.canon.cpu().numpy(), wc))
            else:
                mine = torch.tensor([int(res.entry), int(tail_exit), own_end, n_chunks, int(res.id_base)], dtype=torch.int64, device=dev)
                allv = [torch.empty_like(mine) for _ in range(world)]
                dist.all_gather(allv, mine)
                allv = [t.tolist() for t in allv]
                for r in range(1, world):
                    edges += 1
                    edges_ok = edges_ok and allv[r][0] == allv[r - 1][1] - allv[r - 1][2] and allv[r][4] == allv[r - 1][4] + allv[r - 1][3]
                nmax = max(v[3] for v in allv)
                pad = torch.zeros(nmax, 32, dtype=torch.uint8, device=dev)
                pad[:n_chunks] = res.digests
                gl = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
                dist.gather(pad, gl, dst=0)
                want_canon = torch.empty(sum(v[3] for v in allv), dtype=torch.int64, device=dev)
                if rank == 0:
                    import oracle
                    alld = np.concatenate([g[:allv[r][3]].cpu().numpy() for r, g in enumerate(gl)])
                    wc, _ = oracle.dedup_fast(alld)
                    want_canon.copy_(torch.from_numpy(wc))
                    del gl, alld
                dist.broadcast(want_canon, src=0)
                canon_ok = bool(torch.equal(want_canon[int(res.id_base):int(res.id_base) + n_chunks], res.canon))
                del want_canon, pad
            ok = oc["cuts_equal"] and oc["digests_equal"] and tail_ok and canon_ok
            verify.update({"oracle_equal": bool(red(0 if ok else 1, "sum") == 0) and edges_ok, "edges_checked": edges, "edges_equal": edges_ok,
                           "oracle": {"what": "per rank: oracle.chunk_c + hashlib over the first %.1f GiB of the shard from its entry and over "
                                              "the last 64 MiB before its end (from a GPU cut through the exit) == GPU cuts and digests; "
                                              "entry of rank r == oracle exit of rank r-1; oracle dedup over ALL gathered digests == GPU "
                                              "canon" % (lim / (1 << 30)),
                                      "chunks_checked": int(red(oc["chunks"], "sum")), "bytes_checked": int(red(oc["bytes"], "sum")),
                                      "canon_equal": bool(red(0 if canon_ok else 1, "sum") == 0), "total_s": time.perf_counter() - t_or}})
    # ---- end to end (pinned host shards in, all results out), when the host has the memory for it ----
    e2e = None
    need_gb = world * (n_avail * 1.6) / 1e9
    if not args.no_e2e and world > 1 and need_gb < 0.7 * _mem_available_gb():
        host_in = torch.empty(n_avail, dtype=torch.uint8, pin_memory=True)
        host_in.copy_(d)
        del d, res
        torch.cuda.empty_cache()
        host_out = pipe.host_buffers(n_avail)
        d2h = 0

        def e2e_steps(k):
            nonlocal d2h
            for r in pipe.run_batches([host_in] * k, shard, eof, host=host_out):
                d2h = r.d2h_bytes
        k_e2e = max(1, min(args.steps, 3))
        e2e_steps(1)
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        e2e_steps(k_e2e)
        a1.record()
        barrier()
        ems = red(a0.elapsed_time(a1), "max") / k_e2e
        e2e = {"value": total / (ems * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(red(n_avail, "sum")),
               "d2h_bytes_per_step": int(red(d2h, "sum")), "ms_per_step": ems, "steps": k_e2e,
               "api": "hmse_b200.ShardedIngest.run_batches(pinned host shard buffers, host=pinned result buffers)"}
    elif not args.no_e2e:
        e2e = {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
               "skipped": "needs about %.0f GB of pinned host memory, MemAvailable is %.0f GB" % (need_gb, _mem_available_gb())}
    if rank == 0:
        peak, peak_src = measured_peak()
        line = {"metric": METRIC, "value": total / (ms * 1e-3) / 1e9, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic",
                "config": {"workload": "BASELINE.json configs[3]: ONE %.0f GB high-redundancy stream (CorpusConfig.high_redundancy: 64 %% of "
                                       "the articles are exact duplicates of earlier ones, 16 %% near duplicates) generated on the device, "
                                       "split into %d contiguous byte-range shards; FastCDC + SHA-256 + GLOBAL dedup + DEFLATE of first "
                                       "occurrences" % (args.total_gb, world),
                           "bytes_total": total, "bytes_per_gpu": shard, "parallelism": "byte-range shards, hmse_chunk_sharded + hmse_dedup_global "
                           "(NCCL all-gather of exits, ncclSend/ncclRecv all-to-all of {digest, gid} records by digest prefix)",
                           "l2": "inputs far exceed the 126 MB L2; no explicit flush",
                           "chunks": int(tot_chunks), "unique_chunks": int(uniq_chunks), "unique_chunk_ratio": uniq_chunks / max(1.0, tot_chunks),
                           "unique_bytes": int(uniq_bytes), "exact_duplicate_bytes_frac": 1.0 - uniq_bytes / float(total),
                           "compressed_bytes": int(out_bytes), "data_reduction": total / max(1.0, out_bytes)},
                "stages_ms": stage_ms,
                "exchange": None if xch is None else {"what": "the dedup all-to-all of rank 0, last step: records to owners, answers back",
                                                      "bytes_sent_rank0": xch["bytes_sent"], "bytes_received_rank0": xch["bytes_received"],
                                                      "records_owned_rank0": xch["owned"], "nccl_ms_rank0": xch_ms / args.steps,
                                                      "resync_rounds": xch["rounds"]},
                "roofline": {"bound": "issue", "kernel": "parse_kernel", "achieved": (uniq_bytes + out_bytes) / (max(1e-9, stage_ms["deflate"]) * 1e-3) / 1e9 / world,
                             "peak": peak, "unit": "GB/s", "frac": None, "traffic": None, "peak_source": peak_src,
                             "note": "per-GPU DEFLATE stage bytes / time of rank 0; the per-launch roofline of the dominant kernel is in the configs[1] line"},
                "cpu_baseline": None, "e2e": e2e, "verify": verify, "gpu_launches": int(launches), "clocks": clocks}
        line["roofline"]["frac"] = line["roofline"]["achieved"] / peak
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def run_config5(args):
    """BASELINE.json configs[4]: MinHash (128 permutations, seeds 1..128) + LSH (32 bands x 4 rows) near-duplicate
    detection over ~50 M chunks across the GPUs (write path README.md:1553-1559, MinHash README.md:2578-2597, banding
    README.md:2229-2245).  Every GPU holds its contiguous byte-range shard of ONE stream in HBM (50 M chunks of ~9.4 KB
    over 8 GPUs = 58 GB per GPU: it fits, which a 180 GB part is for), cuts it with boundary resync, signs EVERY chunk,
    sends each band's keys to the band's owner (hmse_lsh_exchange) and the owners sort their bands over all chunks."""
    import ctypes as C
    import numpy as np
    import torch
    import hmse_b200
    from hmse_b200 import corpus as pcorpus
    world, rank, local, dist, ctx, dev, barrier, red = _setup()
    lib = ctx.lib
    cfg, sim = hmse_b200.CDCConfig(), hmse_b200.SimConfig()
    mean_chunk = 9367.0   # bytes per chunk of this corpus (10 GB -> 1 067 542 chunks)
    chunks_total = args.chunks_m * 1e6 * (world / 8.0 if args.chunks_m == 50.0 else 1.0)   # default: 6.25 M chunks per GPU
    total = int(chunks_total * mean_chunk)
    shard = (total // world) & ~15
    eof = rank == world - 1
    lo = rank * shard
    n_avail = (total - lo) if eof else shard + cfg.max_size
    gen = pcorpus.DeviceCorpus(ctx)
    d = gen.generate(n_avail, byte_off=lo)
    torch.cuda.synchronize()
    if world > 1:
        ctx.comm_init()
    simpipe = hmse_b200.ShardedSimilarity(ctx, sim) if world > 1 else None

    def step(timed):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)] if timed else None
        rec = (lambda i: ev[i].record()) if timed else (lambda i: None)
        rec(0)
        if world > 1:
            cuts, entry, id_base, n_total = ctx.chunk_sharded(d, cfg, shard, eof)
        else:
            cuts, entry, id_base = ctx.chunk(d, cfg), 0, 0
            n_total = cuts.numel()
        rec(1)
        sig = ctx.minhash(d, cuts, sim, start0=entry)
        rec(2)
        keys = ctx.lsh_keys(sig, sim)
        rec(3)
        xs = None
        if world > 1:
            owned, _ = ctx.lsh_exchange(keys)
            xs = ctx.exchange_stats()
        else:
            owned = keys
        rec(4)
        band, key, ids = ctx.lsh_buckets(owned.contiguous()) if owned.numel() else (None, None, None)
        rec(5)
        return dict(cuts=cuts, entry=entry, id_base=id_base, n_total=n_total, sig=sig, keys=keys, owned=owned, band=band, key=key,
                    ids=ids, ev=ev, xs=xs)

    out = None
    for _ in range(args.warmup):
        out = None
        torch.cuda.empty_cache()
        out = step(False)
    lib.hmse_timing(ctx.h, 1)
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    l0 = lib.hmse_launch_count(ctx.h)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st_ms = np.zeros(5)
    xms = 0.0
    e0.record()
    for _ in range(args.steps):
        out = None
        out = step(True)
        torch.cuda.synchronize()
        st_ms += np.array([out["ev"][i].elapsed_time(out["ev"][i + 1]) for i in range(5)])
        if out["xs"] is not None:
            xms += out["xs"]["ms"] or 0.0
    e1.record()
    barrier()
    ms = red(e0.elapsed_time(e1), "max") / args.steps
    launches = (lib.hmse_launch_count(ctx.h) - l0) // max(1, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    lib.hmse_timing(ctx.h, 0)
    st_ms /= args.steps
    if args.dump_outputs:
        dump_similarity(args.dump_outputs, out, rank, world)
    n_local = int(out["cuts"].numel())
    n_total = int(out["n_total"])
    own_bytes = int(out["cuts"][-1]) - int(out["entry"]) if n_local else 0
    # ---- checks at full size: (1) a sample of signatures and band keys against the CPU oracle (C MinHash + FNV keys) on
    #      the same chunk bytes, (2) the owner's triples are sorted by (band, key, id) and are as many as chunks x owned
    #      bands, (3) a checksum of checksums: the sum of all keys sent == the sum of all keys in the sorted triples ----
    verify = None
    if not args.no_verify:
        import oracle
        t_or = time.perf_counter()
        rng = np.random.default_rng(11 + rank)
        pick = np.sort(rng.choice(n_local, min(n_local, 256), replace=False))
        cuts_np = out["cuts"].cpu().numpy().view(np.uint64)
        starts_np = np.concatenate([[np.uint64(out["entry"])], cuts_np[:-1]])
        sig_ok = keys_ok = True
        if not args.no_oracle:
            for j in pick.tolist():
                a, b = int(starts_np[j]), int(cuts_np[j])
                raw = d[a:b].cpu().numpy()
                ws = oracle.minhash_c(raw, np.array([b - a], dtype=np.uint64))
                sig_ok = sig_ok and bool(np.array_equal(out["sig"][j].cpu().numpy().view(np.uint32), ws[0]))
                wk = oracle.band_keys(ws)
                keys_ok = keys_ok and bool(np.array_equal(out["keys"][j].cpu().numpy().view(np.uint64), wk[0]))
        sorted_ok, count_ok = True, True
        ksum_sorted = 0
        if out["band"] is not None and out["band"].numel():
            b_, k_, i_ = out["band"], out["key"], out["ids"]
            ku = k_.view(torch.uint64) if hasattr(torch, "uint64") else k_
            # (band, key as unsigned, id) non-decreasing: compare neighbours
            kb = (k_ ^ (-(1 << 63)))     # flip the sign bit: signed order of kb == unsigned order of the key
            le = (b_[:-1] < b_[1:]) | ((b_[:-1] == b_[1:]) & ((kb[:-1] < kb[1:]) | ((kb[:-1] == kb[1:]) & (i_[:-1] < i_[1:]))))
            sorted_ok = bool(le.all())
            count_ok = int(b_.numel()) == n_total * int(out["owned"].shape[1])
            ksum_sorted = int(k_.sum())          # int64 wrap-around sum: a checksum, both sides wrap alike
            del ku, kb, le
        ksum_sent = int(out["keys"].sum())
        tot_sent, tot_sorted = red(float(ksum_sent % (1 << 40)), "sum"), red(float(ksum_sorted % (1 << 40)), "sum")
        checksum_ok = (int(tot_sent) - int(tot_sorted)) % (1 << 40) == 0
        ok = sig_ok and keys_ok and sorted_ok and count_ok
        verify = {"oracle_equal": bool(red(0 if ok else 1, "sum") == 0) and checksum_ok,
                  "signatures_sampled": int(red(pick.size, "sum")) if not args.no_oracle else 0,
                  "signatures_equal": bool(red(0 if sig_ok else 1, "sum") == 0), "band_keys_equal": bool(red(0 if keys_ok else 1, "sum") == 0),
                  "triples_sorted": bool(red(0 if sorted_ok else 1, "sum") == 0), "triples_count_ok": bool(red(0 if count_ok else 1, "sum") == 0),
                  "key_checksum_equal": checksum_ok, "total_s": time.perf_counter() - t_or,
                  "what": "oracle.minhash_c + oracle.band_keys on 256 sampled chunks per rank == GPU signatures and keys; owner triples "
                          "sorted by (band, key, id) and complete; sum of keys sent == sum of keys in the sorted triples (mod 2^40)"}
    if rank == 0:
        props = torch.cuda.get_device_properties(local)
        # alu pipe: 4 schedulers x 16 lanes per cycle per SM; 7.5 alu-pipe instructions per (shingle, seed) evaluation
        # (csrc/minhash.cu: LOP3 x4, SHF x3, half a VIMNMX3), 128 evaluations per byte
        ceil = props.multi_processor_count * 64 * 1965e6 / (128 * 7.5) / 1e9
        mh_gbs = own_bytes / (st_ms[1] * 1e-3) / 1e9
        xs = out["xs"]
        line = {"metric": "similarity GB/s (CDC + MinHash-128 + LSH 32x4 bucketing)", "value": total / (ms * 1e-3) / 1e9, "unit": UNIT,
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
                "config": {"workload": "BASELINE.json configs[4]: MinHash (128 perms) / LSH (32 bands) over %.1f M chunks (%.0f GB of the "
                                       "seed-42 corpus, every chunk signed - no dedup shortcut) across %d B200, one byte-range shard per "
                                       "GPU resident in HBM" % (n_total / 1e6, total / 1e9, world),
                           "chunks": n_total, "chunks_per_s": n_total / (ms * 1e-3), "bytes_total": total, "bytes_per_gpu": shard,
                           "parallelism": "byte-range shards; bands owned by rank b % N; hmse_lsh_exchange (ncclSend/ncclRecv) + per-band radix sort",
                           "l2": "inputs far exceed the 126 MB L2; no explicit flush"},
                "stages_ms_rank0": {"chunk": float(st_ms[0]), "minhash": float(st_ms[1]), "lsh_keys": float(st_ms[2]),
                                    "exchange": float(st_ms[3]), "bucket_sort": float(st_ms[4])},
                "exchange": None if xs is None else {"bytes_sent_rank0": xs["bytes_sent"], "bytes_received_rank0": xs["bytes_received"],
                                                     "nccl_ms_rank0": xms / args.steps,
                                                     "GBps_per_direction_rank0": xs["bytes_sent"] / max(1e-9, xms / args.steps * 1e-3) / 1e9,
                                                     "triples_owned_rank0": int(out["band"].numel()) if out["band"] is not None else 0},
                "roofline": {"bound": "issue", "kernel": "minhash_kernel", "achieved": mh_gbs, "peak": ceil, "unit": "GB/s",
                             "frac": mh_gbs / ceil, "traffic": None,
                             "peak_source": "INT32 alu-pipe issue ceiling: %d SMs x 64 lane-ops/cycle x 1965 MHz / (128 evaluations per byte x "
                                            "7.5 alu-pipe instructions per evaluation); the kernel skips repeated shingles, so it can "
                                            "read above 1.0" % props.multi_processor_count,
                             "hbm_frac": mh_gbs / measured_peak()[0]},
                "cpu_baseline": None, "e2e": None, "verify": verify, "gpu_launches": int(launches), "clocks": clocks}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    args = parse_args()
    # Exactly one line may reach stdout: libraries (NCCL prints its version banner there) are sent
    # to stderr at the file-descriptor level, and the JSON line is written to the saved descriptor.
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    real_stdout = os.fdopen(saved, "w")
    sys.stdout = real_stdout
    try:
        if args.impl == "reference":
            run_reference(args)
        elif args.config == 4:
            run_config4(args)
        elif args.config == 5:
            run_config5(args)
        else:
            run_ours(args)
    finally:
        real_stdout.flush()


if __name__ == "__main__":
    main()
