"""The C ABI driven from C: tests/c_abi/hmse_c_ingest.c (gcc + libcudart + libhmse_b200.so, no Python on its path) runs
the call sequence of INTEGRATION.md; its outputs must equal the Python binding's and the oracle's."""
import os
import subprocess

import numpy as np
import pytest

import oracle
from oracle import corpus

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp_path):
    exe = str(tmp_path / "hmse_c_ingest")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    lib_dir = os.path.join(ROOT, "hmse_b200")
    cmd = ["gcc", "-O1", "-std=c11", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
           os.path.join(ROOT, "tests", "c_abi", "hmse_c_ingest.c"), "-o", exe, "-L", lib_dir, "-lhmse_b200",
           "-L", os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + lib_dir, "-Wl,-rpath," + os.path.join(cuda, "lib64")]
    subprocess.check_call(cmd)
    return exe


@pytest.mark.parametrize("with_dict", [True, False])
def test_c_program_matches_python_binding_and_oracle(ctx, corpus8, tmp_path, with_dict):
    import hmse_b200
    exe = _build(tmp_path)
    data = np.concatenate([corpus8[:3 << 20], corpus8[1 << 20:2 << 20]])
    zd = corpus.zdict() if with_dict else b""
    inp, dic, outp = tmp_path / "in.bin", tmp_path / "dict.bin", tmp_path / "out.bin"
    inp.write_bytes(data.tobytes())
    dic.write_bytes(zd)
    r = subprocess.run([exe, str(inp), str(dic) if with_dict else "-", str(outp)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    buf = outp.read_bytes()
    n, m, total = np.frombuffer(buf, dtype=np.uint64, count=3).tolist()
    o = 24
    cuts = np.frombuffer(buf, dtype=np.uint64, count=n, offset=o); o += 8 * n
    dg = np.frombuffer(buf, dtype=np.uint8, count=32 * n, offset=o).reshape(n, 32); o += 32 * n
    canon = np.frombuffer(buf, dtype=np.int64, count=n, offset=o); o += 8 * n
    sel = np.frombuffer(buf, dtype=np.uint64, count=m, offset=o); o += 8 * m
    offs = np.frombuffer(buf, dtype=np.uint64, count=m + 1, offset=o); o += 8 * (m + 1)
    blob = np.frombuffer(buf, dtype=np.uint8, count=total, offset=o)
    assert o + total == len(buf)
    # the oracle
    wcuts = oracle.chunk_c(data)
    assert np.array_equal(cuts, wcuts)
    wdg = oracle.digest(data, wcuts)
    assert np.array_equal(dg, wdg)
    wcanon, wfirst = oracle.dedup(wdg)
    assert np.array_equal(canon, wcanon) and np.array_equal(sel, np.flatnonzero(wfirst))
    outs = oracle.inflate_all(blob, offs, zd)
    starts = np.concatenate([[0], wcuts[:-1]]).astype(np.int64)
    raw = data.tobytes()
    for k, j in enumerate(sel.astype(np.int64)):
        assert outs[k] == raw[starts[j]:int(wcuts[j])]
    # the Python binding produces the same bytes
    res = hmse_b200.Ingest(ctx, hmse_b200.CDCConfig(), zd).run(ctx.stage(data))
    assert np.array_equal(res.blob.cpu().numpy(), blob) and np.array_equal(res.offsets.cpu().numpy().view(np.uint64), offs)
    assert "kernels launched" in r.stdout


def _build_sharded(tmp_path):
    exe = str(tmp_path / "hmse_c_sharded")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    lib_dir = os.path.join(ROOT, "hmse_b200")
    cmd = ["gcc", "-O1", "-std=gnu11", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
           os.path.join(ROOT, "tests", "c_abi", "hmse_c_sharded.c"), "-o", exe, "-L", lib_dir, "-lhmse_b200",
           "-L", os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + lib_dir, "-Wl,-rpath," + os.path.join(cuda, "lib64")]
    subprocess.check_call(cmd)
    return exe


@pytest.mark.parametrize("world", [1, 2])
def test_c_program_sharded_over_nccl_matches_oracle(corpus8, tmp_path, world):
    """The multi-GPU entry points (hmse_comm_init, hmse_chunk_sharded, hmse_dedup_global, hmse_lsh_exchange) driven from a
    pure C program, one process per GPU: the concatenated shard results equal the oracle over the whole file.  world 1
    runs the same NCCL code path (a one-rank communicator: sends to self) on a one-GPU box; world 2 needs two GPUs."""
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    exe = _build_sharded(tmp_path)
    # duplicates on both sides of every shard edge, and a chunk that straddles it
    data = np.concatenate([corpus8[:3 << 20], corpus8[1 << 20:2 << 20], corpus8[:(2 << 20) + 12345]])
    zd = corpus.zdict()
    inp, dic, prefix = tmp_path / "in.bin", tmp_path / "dict.bin", tmp_path / "out"
    inp.write_bytes(data.tobytes())
    dic.write_bytes(zd)
    env = dict(os.environ)
    # the system libnccl.so.2 or the copy torch ships (a C host has no torch: point the loader at it)
    import glob
    cand = glob.glob(os.path.join(os.path.dirname(torch.__file__), "..", "nvidia", "nccl", "lib"))
    if cand:
        env["LD_LIBRARY_PATH"] = env.get("LD_LIBRARY_PATH", "") + ":" + os.path.abspath(cand[0])
    r = subprocess.run([exe, str(world), str(inp), str(dic), str(prefix)], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    wcuts = oracle.chunk_c(data)
    wdg = oracle.digest(data, wcuts)
    wcanon, wfirst = oracle.dedup(wdg)
    import importlib
    om = importlib.import_module("oracle.minhash")
    _, wkeys, (wb, wk, wi) = om.similarity(data, wcuts, use_c=True)
    starts = np.concatenate([[0], wcuts[:-1]]).astype(np.int64)
    raw = data.tobytes()
    all_cuts, all_dg, all_canon, triples = [], [], [], []
    pos = 0
    for rank in range(world):
        buf = (tmp_path / ("out.%d" % rank)).read_bytes()
        n, m, total, entry, id_base, n_total, lo, nt, rounds = np.frombuffer(buf, dtype=np.uint64, count=9).tolist()
        o = 72
        cuts = np.frombuffer(buf, dtype=np.uint64, count=n, offset=o); o += 8 * n
        dg = np.frombuffer(buf, dtype=np.uint8, count=32 * n, offset=o).reshape(n, 32); o += 32 * n
        canon = np.frombuffer(buf, dtype=np.int64, count=n, offset=o); o += 8 * n
        sel = np.frombuffer(buf, dtype=np.uint64, count=m, offset=o).astype(np.int64); o += 8 * m
        offs = np.frombuffer(buf, dtype=np.uint64, count=m + 1, offset=o); o += 8 * (m + 1)
        blob = np.frombuffer(buf, dtype=np.uint8, count=total, offset=o); o += total
        band = np.frombuffer(buf, dtype=np.uint32, count=nt, offset=o); o += 4 * nt
        key = np.frombuffer(buf, dtype=np.uint64, count=nt, offset=o); o += 8 * nt
        ids = np.frombuffer(buf, dtype=np.uint64, count=nt, offset=o); o += 8 * nt
        assert o == len(buf) and n_total == wcuts.size and id_base == pos and 1 <= rounds <= 3
        assert lo + entry == (int(wcuts[pos - 1]) if pos else 0)          # the shard's first chunk starts at a true cut
        all_cuts.append(cuts + np.uint64(lo))
        all_dg.append(dg)
        all_canon.append(canon)
        # exactly the globally-first chunks of this shard were compressed, and they inflate to their bytes
        assert np.array_equal(sel + pos, np.flatnonzero(wfirst[pos:pos + n]) + pos)
        outs = oracle.inflate_all(blob, offs, zd)
        for k, j in enumerate(sel):
            g = pos + int(j)
            assert outs[k] == raw[starts[g]:int(wcuts[g])]
        triples += list(zip((band.astype(np.int64) * world + rank).tolist(), key.tolist(), ids.tolist()))
        assert set((band.astype(np.int64) * world + rank).tolist()) <= set(range(rank, 32, world))
        pos += n
    assert np.array_equal(np.concatenate(all_cuts), wcuts)
    assert np.array_equal(np.concatenate(all_dg), wdg)
    assert np.array_equal(np.concatenate(all_canon), wcanon)
    assert sorted(triples) == list(zip(wb.tolist(), wk.tolist(), wi.tolist()))
    (tmp_path / "log.txt").write_text(r.stdout)
