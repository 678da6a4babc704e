"""Host side of the hot path: chunk(), digest(), dedup(), compress(), similarity() with the
same names, argument meaning and return layout as the CPU oracle (oracle/__init__.py), served
by the sm_100a kernels behind the C ABI (include/hmse.h).  Spec layers: L2 chunking
README.md:289, L3 digest/dedup README.md:290 + 1288-1292, L1 DEFLATE README.md:288,
L4 MinHash/LSH README.md:291.

Inputs may be host buffers (bytes / numpy) - they are staged to the device and results come back
as numpy arrays, exactly the oracle's return types - or CUDA torch tensors, in which case
results stay on the device as torch tensors.  There is no CPU fallback."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import CdcCfg, HmseError
from .config import CDCConfig, SimConfig

_PAD = 64  # slack after every staged buffer: kernels read whole 16-byte vectors


def _cdc_struct(cfg: CDCConfig) -> CdcCfg:
    s = CdcCfg()
    s.min_size, s.avg_size, s.max_size, s.reserved = cfg.min_size, cfg.avg_size, cfg.max_size, 0
    s.mask_s, s.mask_l = cfg.mask_s, cfg.mask_l
    gear = np.ascontiguousarray(cfg.gear, dtype=np.uint64)  # keep the array alive across the copy
    C.memmove(s.gear, gear.ctypes.data, 2048)
    return s


class Context:
    """One hmse_ctx (device scratch + error text) on one CUDA device."""

    def __init__(self, device: Optional[int] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("hmse_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.cuda.current_device() if device is None else int(device)
        torch.cuda.set_device(self.device)
        torch.cuda.init()
        h = C.c_void_p()
        rc = self.lib.hmse_create(self.device, C.byref(h))
        if rc != 0:
            raise HmseError(rc, "hmse_create failed")
        self.h = h
        self._cdc_cache = {}
        self.comm_world = self.comm_rank = 0   # set by comm_init: this ctx owns an NCCL communicator

    def close(self):
        if getattr(self, "h", None):
            self.lib.hmse_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing ---------------------------------------------------------------------------
    def check(self, rc: int):
        if rc != 0:
            raise HmseError(rc, (self.lib.hmse_last_error(self.h) or b"").decode("utf-8", "replace"))

    @property
    def stream(self) -> C.c_void_p:
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def tdev(self) -> torch.device:
        return torch.device("cuda", self.device)

    def cdc_struct(self, cfg: CDCConfig) -> CdcCfg:
        s = self._cdc_cache.get(cfg)
        if s is None:
            s = self._cdc_cache[cfg] = _cdc_struct(cfg)
        return s

    def empty(self, n: int, dtype) -> torch.Tensor:
        return torch.empty(int(n), dtype=dtype, device=self.tdev)

    def stage(self, data) -> torch.Tensor:
        """uint8 device tensor with 16-byte-aligned storage and >= _PAD readable bytes after it."""
        if isinstance(data, torch.Tensor):
            if data.dtype != torch.uint8 or not data.is_cuda:
                raise TypeError("device input must be a CUDA uint8 tensor")
            data = data.contiguous().view(-1)
            # kernels read whole 16-byte vectors: besides the alignment, _PAD bytes of the same allocation must follow the
            # data (a tensor that ends exactly at the end of its storage could end at the end of a cudaMalloc segment)
            slack = data.untyped_storage().nbytes() - data.storage_offset() - data.numel()
            if data.data_ptr() % 16 == 0 and slack >= _PAD:
                return data
            buf = self.empty(data.numel() + _PAD, torch.uint8)
            buf[:data.numel()].copy_(data)
            return buf[:data.numel()]
        host = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data)
        if host.dtype != np.uint8:
            raise TypeError("data must be uint8")
        buf = self.empty(host.size + _PAD, torch.uint8)
        if host.size:
            buf[:host.size].copy_(torch.from_numpy(host.reshape(-1).copy() if not host.flags.writeable else host.reshape(-1)))
        return buf[:host.size]

    def stage_u64(self, x) -> torch.Tensor:
        """int64 device tensor holding uint64 bit patterns."""
        if isinstance(x, torch.Tensor):
            if x.dtype not in (torch.int64, torch.uint64) or not x.is_cuda:
                raise TypeError("device cuts must be a CUDA int64/uint64 tensor")
            return x.contiguous().view(torch.int64)
        a = np.ascontiguousarray(x, dtype=np.uint64).view(np.int64)
        return torch.from_numpy(a.copy()).to(self.tdev)

    # -- L2 -------------------------------------------------------------------------------
    def chunk(self, d: torch.Tensor, cfg: CDCConfig) -> torch.Tensor:
        n = d.numel()
        cap = n // cfg.min_size + 2
        cuts = self.empty(cap, torch.int64)
        nc = C.c_uint64(0)
        self.check(self.lib.hmse_chunk(self.h, d.data_ptr(), n, C.byref(self.cdc_struct(cfg)), cuts.data_ptr(), cap,
                                       C.byref(nc), self.stream))
        return cuts[:nc.value]

    def chunk_files(self, d: torch.Tensor, file_off: torch.Tensor, cfg: CDCConfig):
        """(cuts int64, file_chunk int64[F+1]): file f = d[file_off[f]:file_off[f+1]] chunked on its own (hmse_chunk_files);
        file_off is an int64 device tensor of F+1 offsets from 0 to d.numel()."""
        n, nf = d.numel(), file_off.numel() - 1
        if nf < 0:
            raise ValueError("file_off needs at least one entry")
        cap = n // cfg.min_size + nf + 1
        cuts = self.empty(cap, torch.int64)
        fc = self.empty(nf + 1, torch.int64)
        nc = C.c_uint64(0)
        self.check(self.lib.hmse_chunk_files(self.h, d.data_ptr(), n, file_off.data_ptr(), nf, C.byref(self.cdc_struct(cfg)),
                                             cuts.data_ptr(), cap, C.byref(nc), fc.data_ptr(), self.stream))
        return cuts[:nc.value], fc

    def chunk_scan(self, d: torch.Tensor, cfg: CDCConfig):
        self.check(self.lib.hmse_chunk_scan(self.h, d.data_ptr(), d.numel(), C.byref(self.cdc_struct(cfg)), self.stream))

    def chunk_candidates(self, n: int):
        """(bits_s, bits_l) int64 tensors: candidate bitmaps of the last chunk_scan over n bytes."""
        words = (n + 63) // 64
        bs, bl = self.empty(words, torch.int64), self.empty(words, torch.int64)
        self.check(self.lib.hmse_chunk_candidates(self.h, bs.data_ptr(), bl.data_ptr(), words, self.stream))
        return bs, bl

    def chunk_resolve(self, d: torch.Tensor, cfg: CDCConfig, n_own: int, eof: bool, entry: int):
        """Returns (cuts int64 tensor, exit offset).  Requires a prior chunk_scan(d, cfg)."""
        n = d.numel()
        own = n if eof else n_own
        cap = own // cfg.min_size + 2
        cuts = self.empty(cap, torch.int64)
        nc, ex = C.c_uint64(0), C.c_uint64(0)
        self.check(self.lib.hmse_chunk_resolve(self.h, d.data_ptr(), n_own, n, int(eof), entry, cuts.data_ptr(), cap,
                                               C.byref(nc), C.byref(ex), self.stream))
        return cuts[:nc.value], ex.value

    # -- multi-GPU: the exchange steps behind the C ABI (csrc/comm.cu, NCCL) ------------------------
    def comm_init(self, group=None) -> None:
        """Creates this context's NCCL communicator over the ranks of a torch.distributed group (default: the world
        group): rank 0 draws the ncclUniqueId, torch.distributed carries its 128 bytes, every rank calls hmse_comm_init.
        torch.distributed is only the side channel here - the data path collectives are issued by the library."""
        import torch.distributed as dist
        if self.comm_world:
            return
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        uid = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            buf = (C.c_uint8 * 128)()
            rc = self.lib.hmse_comm_unique_id(buf)
            if rc != 0:
                raise HmseError(rc, "hmse_comm_unique_id failed (is libnccl.so.2 loadable?)")
            uid = torch.frombuffer(bytearray(buf), dtype=torch.uint8).clone()
        on_gpu = dist.get_backend(group) == "nccl"
        t = uid.to(self.tdev) if on_gpu else uid
        dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        raw = bytes(t.cpu().numpy().tobytes())
        self.check(self.lib.hmse_comm_init(self.h, raw, world, rank))
        self.comm_world, self.comm_rank = world, rank

    def chunk_sharded(self, d: torch.Tensor, cfg: CDCConfig, n_own: int, eof: bool):
        """(cuts, entry, id_base, n_total) of this rank's byte-range shard of one stream (hmse_chunk_sharded)."""
        n = d.numel()
        own = n if eof else n_own
        cap = own // cfg.min_size + 2
        cuts = self.empty(cap, torch.int64)
        nc, en, ib, nt = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        self.check(self.lib.hmse_chunk_sharded(self.h, None, d.data_ptr(), n_own, n, int(eof), C.byref(self.cdc_struct(cfg)),
                                               cuts.data_ptr(), cap, C.byref(nc), C.byref(en), C.byref(ib), C.byref(nt),
                                               self.stream))
        return cuts[:nc.value], en.value, ib.value, nt.value

    def dedup_global(self, digests: torch.Tensor, id_base: int):
        """(canon int64[n] of GLOBAL ids, is_first uint8[n]) over every rank's digests (hmse_dedup_global)."""
        n = digests.shape[0]
        canon = self.empty(max(n, 1), torch.int64)
        first = self.empty(max(n, 1), torch.uint8)
        self.check(self.lib.hmse_dedup_global(self.h, None, digests.data_ptr(), n, id_base, canon.data_ptr(), first.data_ptr(),
                                              self.stream))
        return canon[:n], first[:n]

    def lsh_exchange(self, keys: torch.Tensor):
        """(owned int64 [N_total, bands_owned], id_base): the owned bands' keys of every chunk of the stream."""
        n, bands = int(keys.shape[0]), int(keys.shape[1])
        nt, ib, bo = C.c_uint64(0), C.c_uint64(0), C.c_uint32(0)
        keys = keys.contiguous()
        self.check(self.lib.hmse_lsh_exchange(self.h, None, keys.data_ptr(), n, bands, None, 0, C.byref(nt), C.byref(ib),
                                              C.byref(bo), self.stream))
        owned = self.empty(max(1, nt.value * bo.value), torch.int64)
        self.check(self.lib.hmse_lsh_exchange(self.h, None, keys.data_ptr(), n, bands, owned.data_ptr(), nt.value, C.byref(nt),
                                              C.byref(ib), C.byref(bo), self.stream))
        return owned[:nt.value * bo.value].view(nt.value, bo.value), ib.value

    def allgather4(self, a: int, b: int = 0, c: int = 0, d: int = 0):
        """[[a, b, c, d] of rank 0, ... of rank world-1] (hmse_allgather_u64: one collective, one host round trip)."""
        w = self.comm_world
        vals = (C.c_uint64 * 4)(int(a), int(b), int(c), int(d))
        out = (C.c_uint64 * (4 * w))()
        self.check(self.lib.hmse_allgather_u64(self.h, None, vals, out, self.stream))
        return [[int(out[4 * r + q]) for q in range(4)] for r in range(w)]

    def delta_heads(self, band: torch.Tensor, key: torch.Tensor, ids: torch.Tensor, n: int, bands: int) -> torch.Tensor:
        """heads int32 [n, bands] (uint32 bit patterns): first id of every chunk's bucket, from sorted triples."""
        heads = self.empty(max(1, n * bands), torch.int32)
        self.check(self.lib.hmse_delta_heads(self.h, band.data_ptr(), key.data_ptr(), ids.data_ptr(), n, bands, 0, None,
                                             heads.data_ptr(), self.stream))
        return heads[:n * bands].view(n, bands)

    def delta_votes(self, heads: torch.Tensor, id_base: int, min_votes: int, root_all: Optional[torch.Tensor] = None):
        """pass 0 (root_all None): root flags uint8[n] of this rank's chunks; pass 1: base int64[n] (ids in the heads' space)."""
        n, bands = int(heads.shape[0]), int(heads.shape[1])
        heads = heads.contiguous()
        if root_all is None:
            root = self.empty(max(1, n), torch.uint8)
            self.check(self.lib.hmse_delta_votes(self.h, heads.data_ptr(), n, bands, id_base, min_votes, 0, root.data_ptr(), None,
                                                 None, self.stream))
            return root[:n]
        base = self.empty(max(1, n), torch.int64)
        self.check(self.lib.hmse_delta_votes(self.h, heads.data_ptr(), n, bands, id_base, min_votes, 1, None, root_all.data_ptr(),
                                             base.data_ptr(), self.stream))
        return base[:n]

    def alltoallv(self, send: torch.Tensor, send_counts, elem_bytes: int):
        """(recv uint8 tensor, recv_counts list): `send` (uint8, elements of elem_bytes grouped by destination rank,
        send_counts[world] of them per rank) through hmse_alltoallv."""
        w = self.comm_world
        sc = (C.c_uint64 * w)(*[int(c) for c in send_counts])
        rc = (C.c_uint64 * w)()
        send = send.contiguous()
        self.check(self.lib.hmse_alltoallv(self.h, None, send.data_ptr() if send.numel() else None, sc, None, rc, elem_bytes, 0,
                                           self.stream))
        total = sum(int(x) for x in rc)
        recv = self.empty(total * elem_bytes + _PAD, torch.uint8)     # slack: receivers may read whole words past the end
        self.check(self.lib.hmse_alltoallv(self.h, None, send.data_ptr() if send.numel() else None, sc, recv.data_ptr(), rc,
                                           elem_bytes, total, self.stream))
        return recv[:total * elem_bytes], [int(x) for x in rc]

    def exchange_stats(self):
        """{bytes_sent, bytes_received, owned, contributed, rounds, ms} of the last exchange (ms only with hmse_timing on)."""
        out = (C.c_uint64 * 4)()
        rounds = C.c_int(0)
        self.check(self.lib.hmse_exchange_stats(self.h, out, C.byref(rounds)))
        f = C.c_float(0)
        ms = f.value if self.lib.hmse_timing_ms(self.h, 10, C.byref(f)) == 0 else None
        return {"bytes_sent": int(out[0]), "bytes_received": int(out[1]), "owned": int(out[2]), "contributed": int(out[3]),
                "rounds": int(rounds.value), "ms": ms}

    # -- L3 -------------------------------------------------------------------------------
    def digest(self, d: torch.Tensor, cuts: torch.Tensor, start0: int = 0) -> torch.Tensor:
        m = cuts.numel()
        out = self.empty(m * 32, torch.uint8)
        self.check(self.lib.hmse_digest(self.h, d.data_ptr(), start0, cuts.data_ptr(), m, out.data_ptr(), self.stream))
        return out.view(m, 32)

    def dedup(self, digests: torch.Tensor):
        m = digests.shape[0]
        canon = self.empty(m, torch.int64)
        first = self.empty(m, torch.uint8)
        self.check(self.lib.hmse_dedup(self.h, digests.data_ptr(), m, canon.data_ptr(), first.data_ptr(), self.stream))
        return canon, first.view(torch.bool)

    # -- L1 -------------------------------------------------------------------------------
    def compress(self, d: torch.Tensor, cuts: torch.Tensor, select: Optional[torch.Tensor], zdict: Optional[torch.Tensor],
                 level: int = 6, start0: int = 0, out_cap: Optional[int] = None, out: Optional[torch.Tensor] = None):
        """(blob, offsets).  `out` (uint8 device tensor) receives the blob when it is large enough; otherwise a
        tensor of the required size is allocated (input bytes + per-chunk slack bounds any stream)."""
        m = cuts.numel() if select is None else select.numel()
        offsets = self.empty(m + 1, torch.int64)
        total = C.c_uint64(0)
        zp = zdict.data_ptr() if zdict is not None and zdict.numel() else None
        zl = zdict.numel() if zdict is not None else 0
        sp = select.data_ptr() if select is not None else None
        cap = out.numel() if out is not None else (int(out_cap) if out_cap is not None else 0)
        if out is None and cap:
            out = self.empty(cap, torch.uint8)
        # without a buffer the first call only sizes the result (the streams stay staged in the ctx) and the pack
        # writes a blob of exactly that size; a buffer that turns out too small is replaced the same way
        rc = self.lib.hmse_compress(self.h, d.data_ptr(), start0, cuts.data_ptr(), sp, m, zp, zl, level,
                                    out.data_ptr() if out is not None else None, cap, offsets.data_ptr(), C.byref(total), self.stream)
        if (out is None and rc == 0) or (rc == _lib.HMSE_E_CAPACITY and total.value > cap):
            out = self.empty(max(1, total.value), torch.uint8)
            rc = self.lib.hmse_compress_pack(self.h, offsets.data_ptr(), m, out.data_ptr(), out.numel(), self.stream)
        self.check(rc)
        return out[:total.value], offsets

    def compress_known(self, src, d: torch.Tensor, cuts: torch.Tensor, digests: torch.Tensor, select: Optional[torch.Tensor],
                       zdict: Optional[torch.Tensor], level: int = 6, start0: int = 0, out: Optional[torch.Tensor] = None):
        """compress() against an opened archive (hmse_compress_known): `src` is the archive's _lib.ComposeSrc, `digests` the
        SHA-256 of every chunk.  Streams the archive holds are copied from it, the others compressed; blob and offsets
        equal compress()'s.  Returns (blob, offsets, known int64[m]: source slot copied or -1, stats4 = [streams copied,
        bytes copied, streams compressed, raw bytes compressed])."""
        m = cuts.numel() if select is None else select.numel()
        offsets = self.empty(m + 1, torch.int64)
        known = self.empty(max(m, 1), torch.int64)
        total, st4 = C.c_uint64(0), (C.c_uint64 * 4)()
        zp = zdict.data_ptr() if zdict is not None and zdict.numel() else None
        zl = zdict.numel() if zdict is not None else 0
        sp = select.data_ptr() if select is not None else None
        cap = out.numel() if out is not None else 0
        # as compress(): without a buffer the first call plans and sizes, the pack writes a blob of exactly that size
        rc = self.lib.hmse_compress_known(self.h, C.byref(src), d.data_ptr(), start0, cuts.data_ptr(), digests.data_ptr(), sp, m,
                                          zp, zl, level, out.data_ptr() if out is not None else None, cap, offsets.data_ptr(),
                                          C.byref(total), known.data_ptr(), st4, self.stream)
        if (out is None and rc == 0) or (rc == _lib.HMSE_E_CAPACITY and total.value > cap):
            out = self.empty(max(1, total.value), torch.uint8)
            rc = self.lib.hmse_compress_known_pack(self.h, offsets.data_ptr(), m, out.data_ptr(), out.numel(), self.stream)
        self.check(rc)
        return out[:total.value], offsets, known[:m], [int(x) for x in st4]

    def inflate(self, blob: torch.Tensor, offsets: torch.Tensor, out_offsets: torch.Tensor, zdict: Optional[torch.Tensor]):
        """(out uint8[out_offsets[-1]], status int32[m], n_bad): every stream inflated on the device."""
        m = offsets.numel() - 1
        total = int(out_offsets[-1]) if out_offsets.numel() else 0
        out = self.empty(total + _PAD, torch.uint8)[:total]
        status = self.empty(max(m, 1), torch.int32)[:m]
        bad = C.c_uint64(0)
        zp = zdict.data_ptr() if zdict is not None and zdict.numel() else None
        zl = zdict.numel() if zdict is not None else 0
        self.check(self.lib.hmse_inflate(self.h, blob.data_ptr(), offsets.data_ptr(), m, zp, zl, out.data_ptr(),
                                         out_offsets.data_ptr(), status.data_ptr(), C.byref(bad), self.stream))
        return out, status, int(bad.value)

    # -- L4 -------------------------------------------------------------------------------
    def minhash(self, d: torch.Tensor, cuts: torch.Tensor, cfg: SimConfig, start0: int = 0,
                select: Optional[torch.Tensor] = None) -> torch.Tensor:
        """sig int32[m, n_perm] of every chunk, or (select: int64 chunk indices) of the selected chunks only."""
        seeds = torch.from_numpy(cfg.seed_array.view(np.int32).copy()).to(self.tdev)
        if select is not None:
            m = select.numel()
            sig = self.empty(m * cfg.n_perm, torch.int32)
            self.check(self.lib.hmse_minhash_select(self.h, d.data_ptr(), start0, cuts.data_ptr(), select.data_ptr(), m,
                                                    seeds.data_ptr(), cfg.n_perm, sig.data_ptr(), self.stream))
            return sig.view(m, cfg.n_perm)
        m = cuts.numel()
        sig = self.empty(m * cfg.n_perm, torch.int32)
        self.check(self.lib.hmse_minhash(self.h, d.data_ptr(), start0, cuts.data_ptr(), m, seeds.data_ptr(), cfg.n_perm,
                                         sig.data_ptr(), self.stream))
        return sig.view(m, cfg.n_perm)

    def lsh_keys(self, sig: torch.Tensor, cfg: SimConfig) -> torch.Tensor:
        m = sig.shape[0]
        keys = self.empty(m * cfg.bands, torch.int64)
        self.check(self.lib.hmse_lsh_keys(self.h, sig.data_ptr(), m, cfg.bands, cfg.rows, keys.data_ptr(), self.stream))
        return keys.view(m, cfg.bands)

    def lsh_buckets(self, keys: torch.Tensor, id_base: int = 0):
        m, b = keys.shape
        band = self.empty(m * b, torch.int32)
        key = self.empty(m * b, torch.int64)
        ids = self.empty(m * b, torch.int64)
        self.check(self.lib.hmse_lsh_buckets(self.h, keys.data_ptr(), m, b, id_base, band.data_ptr(), key.data_ptr(),
                                             ids.data_ptr(), self.stream))
        return band, key, ids

    def delta_bases(self, band: torch.Tensor, key: torch.Tensor, ids: torch.Tensor, n: int, bands: int,
                    is_first: torch.Tensor, min_votes: int = 4, id_base: int = 0) -> torch.Tensor:
        """base int64[n]: the root chunk each first-occurrence chunk would be delta-coded against, or -1."""
        base = self.empty(n, torch.int64)
        f = is_first.view(torch.uint8) if is_first.dtype == torch.bool else is_first
        self.check(self.lib.hmse_delta_bases(self.h, band.data_ptr(), key.data_ptr(), ids.data_ptr(), n, bands, id_base,
                                             f.contiguous().data_ptr(), min_votes, base.data_ptr(), self.stream))
        return base

    def delta_encode(self, d: torch.Tensor, cuts: torch.Tensor, base: torch.Tensor, start0: int = 0, ext=None):
        """(blob, offsets int64[n+1]); `base` is updated in place (-1 where the 20 % rule rejected the delta).
        ext = (ext_data uint8 with slack, ext_off int64[n_ext + 1]): base values >= n name external bases (chunks of
        another shard), see hmse_delta_encode_ext."""
        n = cuts.numel()
        ep, eo, ne = (ext[0].data_ptr(), ext[1].data_ptr(), ext[1].numel() - 1) if ext is not None else (None, None, 0)
        offsets = self.empty(n + 1, torch.int64)
        total = C.c_uint64(0)
        # kept deltas are a fraction of a percent of the stream (0.14 % on the wiki corpus): 1/64 of it rarely needs the
        # retry, which repeats the whole encode
        out_cap = max(1 << 20, int(d.numel()) // 64)
        for _ in range(2):
            out = self.empty(out_cap + _PAD, torch.uint8)
            rc = self.lib.hmse_delta_encode_ext(self.h, d.data_ptr(), start0, cuts.data_ptr(), n, base.data_ptr(), ep, eo, ne,
                                                out.data_ptr(), out_cap, offsets.data_ptr(), C.byref(total), self.stream)
            if rc == _lib.HMSE_E_CAPACITY and total.value > out_cap:
                out_cap = int(total.value)  # the encode is deterministic: the retry reproduces it
                continue
            self.check(rc)
            return out[:total.value], offsets
        raise HmseError(_lib.HMSE_E_CAPACITY, "hmse_delta_encode: capacity retry failed")

    def delta_apply(self, blob: torch.Tensor, offsets: torch.Tensor, base_data: torch.Tensor, base_off: torch.Tensor,
                    base_len: torch.Tensor, out_offsets: torch.Tensor):
        """(out uint8, status int32[m], n_bad)."""
        m = offsets.numel() - 1
        total = int(out_offsets[-1]) if out_offsets.numel() else 0
        out = self.empty(total + _PAD, torch.uint8)[:total]
        status = self.empty(max(m, 1), torch.int32)[:m]
        bad = C.c_uint64(0)
        self.check(self.lib.hmse_delta_apply(self.h, blob.data_ptr(), offsets.data_ptr(), m, base_data.data_ptr(),
                                             base_data.numel(), base_off.data_ptr(), base_len.data_ptr(), out.data_ptr(), out_offsets.data_ptr(),
                                             status.data_ptr(), C.byref(bad), self.stream))
        return out, status, int(bad.value)


_contexts = {}


def default_context(device: Optional[int] = None) -> Context:
    if not torch.cuda.is_available():
        raise RuntimeError("hmse_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    dev = torch.cuda.current_device() if device is None else int(device)
    ctx = _contexts.get(dev)
    if ctx is None:
        ctx = _contexts[dev] = Context(dev)
    return ctx


def _is_dev(x) -> bool:
    return isinstance(x, torch.Tensor) and x.is_cuda


def _np_u64(t: torch.Tensor) -> np.ndarray:
    return t.cpu().numpy().view(np.uint64)


# ---- the oracle-shaped API --------------------------------------------------------------------

def chunk(data, cfg: CDCConfig = CDCConfig(), ctx: Optional[Context] = None):
    """cuts: uint64[n] exclusive end offsets, strictly increasing, cuts[-1] == len(data)."""
    ctx = ctx or default_context()
    cuts = ctx.chunk(ctx.stage(data), cfg)
    return cuts if _is_dev(data) else _np_u64(cuts)


def file_offsets(sizes, n: int, ctx: Context) -> torch.Tensor:
    """int64 device tensor [F+1]: 0, then the running sum of the file sizes (which must add up to n)."""
    if _is_dev(sizes):
        sz = sizes.to(torch.int64)
        off = torch.cat([torch.zeros(1, dtype=torch.int64, device=sz.device), torch.cumsum(sz, 0)])
        return off.to(ctx.tdev)
    sz = np.asarray(sizes, dtype=np.int64).reshape(-1)
    if (sz < 0).any():
        raise ValueError("file sizes must be >= 0")
    off = np.concatenate([[0], np.cumsum(sz)]).astype(np.int64)
    if int(off[-1]) != n:
        raise ValueError("file sizes add up to %d, the data has %d bytes" % (int(off[-1]), n))
    return torch.from_numpy(off).to(ctx.tdev)


def chunk_files(data, sizes, cfg: CDCConfig = CDCConfig(), ctx: Optional[Context] = None):
    """Many files in one call: `data` holds the files back to back, `sizes[f]` bytes each (0 allowed).  Every file is
    chunked on its own, exactly as chunk() chunks it alone.  Returns (cuts uint64[n], file_chunk uint64[F+1]): one chunk
    list over the whole buffer (absolute offsets), and the index of each file's first chunk (an empty file shares the
    index of the next file; file_chunk[F] = n).  Host input gives numpy arrays, CUDA input CUDA tensors."""
    ctx = ctx or default_context()
    d = ctx.stage(data)
    cuts, fc = ctx.chunk_files(d, file_offsets(sizes, d.numel(), ctx), cfg)
    return (cuts, fc) if _is_dev(data) else (_np_u64(cuts), _np_u64(fc))


def digest(data, cuts, start0: int = 0, ctx: Optional[Context] = None):
    """uint8[n, 32]: SHA-256 of every raw chunk."""
    ctx = ctx or default_context()
    out = ctx.digest(ctx.stage(data), ctx.stage_u64(cuts), start0)
    return out if _is_dev(data) else out.cpu().numpy()


def dedup(digests, ctx: Optional[Context] = None):
    """(canon int64[n], is_first bool[n]): canon[i] = first index with the same digest."""
    ctx = ctx or default_context()
    dev = _is_dev(digests)
    dg = digests if dev else torch.from_numpy(np.ascontiguousarray(digests, dtype=np.uint8).reshape(-1, 32)).to(ctx.tdev)
    canon, first = ctx.dedup(dg.contiguous())
    return (canon, first) if dev else (canon.cpu().numpy(), first.cpu().numpy())


def compress(data, cuts, select, zdict: bytes = b"", level: int = 6, start0: int = 0, ctx: Optional[Context] = None):
    """(blob uint8[...], offsets uint64[m+1]); slice j is one zlib stream (FDICT when zdict)."""
    ctx = ctx or default_context()
    dev = _is_dev(data)
    d = ctx.stage(data)
    sel = None if select is None else ctx.stage_u64(select)
    zd = ctx.stage(zdict) if not isinstance(zdict, torch.Tensor) else zdict
    blob, offs = ctx.compress(d, ctx.stage_u64(cuts), sel, zd, level, start0)
    return (blob, offs) if dev else (blob.cpu().numpy(), _np_u64(offs))


def inflate(blob, offsets, sizes, zdict: bytes = b"", ctx: Optional[Context] = None):
    """The read path: (raw uint8[sum(sizes)], status int32[m]).  Stream j inflates to `sizes[j]` bytes at
    offset sum(sizes[:j]); status[j] == 0 iff it is well formed and its Adler-32 (and DICTID) check out."""
    ctx = ctx or default_context()
    dev = _is_dev(blob)
    b = ctx.stage(blob)
    offs = ctx.stage_u64(offsets)
    sz = np.ascontiguousarray(sizes.cpu().numpy() if isinstance(sizes, torch.Tensor) else sizes, dtype=np.uint64)
    oo = np.concatenate([[np.uint64(0)], np.cumsum(sz, dtype=np.uint64)])
    zd = ctx.stage(zdict) if not isinstance(zdict, torch.Tensor) else zdict
    out, status, _ = ctx.inflate(b, offs, ctx.stage_u64(oo), zd)
    return (out, status) if dev else (out.cpu().numpy(), status.cpu().numpy())


def compress_bound(n: int) -> int:
    """Worst-case bytes of one zlib stream for a chunk of n bytes (hmse_compress_bound)."""
    return int(_lib.load().hmse_compress_bound(int(n)))


def similarity(data, cuts, cfg: SimConfig = SimConfig(), start0: int = 0, ctx: Optional[Context] = None):
    """(sig uint32[n, n_perm], keys uint64[n, bands], (band u32, key u64, id u64) sorted)."""
    ctx = ctx or default_context()
    dev = _is_dev(data)
    d = ctx.stage(data)
    sig = ctx.minhash(d, ctx.stage_u64(cuts), cfg, start0)
    keys = ctx.lsh_keys(sig, cfg)
    band, key, ids = ctx.lsh_buckets(keys)
    if dev:
        return sig, keys, (band, key, ids)
    return (sig.cpu().numpy().view(np.uint32), _np_u64(keys),
            (band.cpu().numpy().view(np.uint32), _np_u64(key), _np_u64(ids)))


def delta(data, cuts, keys, is_first, min_votes: int = 4, start0: int = 0, ctx: Optional[Context] = None):
    """L4 delta coding (README.md:1328, 2160-2198): (base int64[n], blob uint8[...], offsets uint64[n+1]).
    Chunk i is stored as a delta against chunk base[i] iff offsets[i+1] > offsets[i]; base[i] is -1 where no
    delta is kept.  `keys` are the band keys of similarity() (uint64[n, bands], bands <= 32)."""
    ctx = ctx or default_context()
    dev = _is_dev(data)
    d = ctx.stage(data)
    c = ctx.stage_u64(cuts)
    k = keys if _is_dev(keys) else torch.from_numpy(np.ascontiguousarray(keys, dtype=np.uint64).view(np.int64).copy()).to(ctx.tdev)
    f = is_first if _is_dev(is_first) else torch.from_numpy(np.ascontiguousarray(is_first, dtype=np.uint8).copy()).to(ctx.tdev)
    n, bands = k.shape
    band, key, ids = ctx.lsh_buckets(k.contiguous())
    base = ctx.delta_bases(band, key, ids, n, bands, f, min_votes)
    blob, offs = ctx.delta_encode(d, c, base, start0)
    return (base, blob, offs) if dev else (base.cpu().numpy(), blob.cpu().numpy(), _np_u64(offs))


def delta_apply(blob, offsets, bases, base_sizes, sizes, ctx: Optional[Context] = None):
    """The L4 read path: delta j applied to raw base j (the bases concatenated in `bases`, `base_sizes[j]` bytes
    each) gives `sizes[j]` bytes; returns (raw uint8[sum(sizes)], status int32[m])."""
    ctx = ctx or default_context()
    dev = _is_dev(blob)
    b = ctx.stage(blob)
    offs = ctx.stage_u64(offsets)
    bd = ctx.stage(bases)
    to_np = lambda x: np.ascontiguousarray(x.cpu().numpy() if isinstance(x, torch.Tensor) else x)  # noqa: E731
    bs = to_np(base_sizes).astype(np.uint64)
    bo = np.concatenate([[np.uint64(0)], np.cumsum(bs, dtype=np.uint64)])[:-1]
    sz = to_np(sizes).astype(np.uint64)
    oo = np.concatenate([[np.uint64(0)], np.cumsum(sz, dtype=np.uint64)])
    bl = torch.from_numpy(bs.astype(np.uint32).view(np.int32).copy()).to(ctx.tdev)
    out, status, _ = ctx.delta_apply(b, offs, bd, ctx.stage_u64(bo), bl, ctx.stage_u64(oo))
    return (out, status) if dev else (out.cpu().numpy(), status.cpu().numpy())
