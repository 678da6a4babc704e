"""hmse_inflate against stock zlib on every RFC 1950 / 1951 feature, valid and malformed (tests/model/inflate_cases.py):
the decoder must accept exactly the streams `zlib_verdict` accepts, and write zlib's bytes for them.  Corpus text from
a real encoder reaches only a narrow part of the format; these streams reach the code shapes at and past the direct
lookup widths, degenerate and incomplete codes, header extremes, every length and distance boundary, the preset
dictionary's first byte, stored blocks at every bit phase, the trailer and the damaged forms of three small streams.

Each group is one call with its cases shuffled, a spacer stream between every two of them: a spacer's stream has a
bad CMF, so the kernel rejects it before writing, and its 64-byte output range must still hold the canary afterwards."""
import ctypes as C
import time

import numpy as np
import pytest

from tests.model import inflate_cases

pytestmark = pytest.mark.gpu

CANARY = 0xA5
SPACER = b"\x77\x01" + bytes(14)   # CM 7: rejected on the header, before any output
SPACER_OUT = 64


def _run_group(ctx, group, seed):
    """(status per case, bytes per case, spacer ranges intact, n_bad) of one hmse_inflate call over the group."""
    import torch
    cases = group.cases
    order = np.random.default_rng(seed).permutation(len(cases))
    streams, outs, kinds = [SPACER], [SPACER_OUT], [-1]
    for k in order.tolist():
        streams += [cases[k].stream, SPACER]
        outs += [cases[k].out_len, SPACER_OUT]
        kinds += [k, -1]
    offs = np.concatenate([[0], np.cumsum([len(s) for s in streams])]).astype(np.uint64)
    oo = np.concatenate([[0], np.cumsum(outs)]).astype(np.uint64)
    blob = ctx.stage(np.frombuffer(b"".join(streams), np.uint8))
    d_offs, d_oo = ctx.stage_u64(offs), ctx.stage_u64(oo)
    total = int(oo[-1])
    out = torch.full((total + SPACER_OUT,), CANARY, dtype=torch.uint8, device=ctx.tdev)   # a canary tail as well
    status = torch.full((len(streams),), -1, dtype=torch.int32, device=ctx.tdev)
    zd = ctx.stage(np.frombuffer(group.zd, np.uint8)) if group.zd else None
    bad = C.c_uint64(0)
    ctx.check(ctx.lib.hmse_inflate(ctx.h, blob.data_ptr(), d_offs.data_ptr(), len(streams),
                                   zd.data_ptr() if zd is not None else None, len(group.zd), out.data_ptr(),
                                   d_oo.data_ptr(), status.data_ptr(), C.byref(bad), ctx.stream))
    torch.cuda.synchronize()
    out, status = out.cpu().numpy(), status.cpu().numpy()
    got_status, got_bytes, spacers_ok = [None] * len(cases), [None] * len(cases), True
    for i, k in enumerate(kinds):
        rng = out[int(oo[i]):int(oo[i + 1])]
        if k < 0:
            spacers_ok &= bool(status[i] != 0) and bool((rng == CANARY).all())
        else:
            got_status[k], got_bytes[k] = int(status[i]), rng.tobytes()
    spacers_ok &= bool((out[total:] == CANARY).all())
    return got_status, got_bytes, spacers_ok, int(bad.value), len(cases) + 1


def _explain(case, got, want):
    """Where the GPU's bytes first differ from zlib's, and what the stream holds."""
    i = next((i for i in range(min(len(got), len(want))) if got[i] != want[i]), min(len(got), len(want)))
    return "output byte %d of %d differs (gpu %s, zlib %s); %s" % (
        i, len(want), got[i] if i < len(got) else "-", want[i] if i < len(want) else "-", inflate_cases.describe(case.stream))


@pytest.mark.parametrize("family", list(inflate_cases.FAMILIES))
def test_decoder_agrees_with_zlib(ctx, family):
    t0 = time.time()
    bad, n_streams, n_accept = [], 0, 0
    for gi, group in enumerate(inflate_cases.FAMILIES[family]()):
        status, outs, spacers_ok, n_bad, n_spacers = _run_group(ctx, group, seed=1000 + gi)
        rejected = 0
        for case, st, got in zip(group.cases, status, outs):
            want = inflate_cases.zlib_verdict(case.stream, group.zd, case.out_len)
            rejected += st != 0
            n_accept += want is not None
            tag = "%s / %s" % (group.name, case.name)
            if (want is None) != (st != 0):
                bad.append("%s: gpu status %d, zlib %s - %s" % (tag, st, "rejects it" if want is None else "accepts it",
                                                               inflate_cases.describe(case.stream)))
            elif want is not None and got != want:
                bad.append("%s: %s" % (tag, _explain(case, got, want)))
            elif case.status is not None and st != case.status:
                bad.append("%s: status %d, the kernel documents %d" % (tag, st, case.status))
        assert spacers_ok, "%s: a spacer stream was accepted or its output range was written" % group.name
        assert n_bad == rejected + n_spacers, "%s: n_bad %d, %d rejected streams" % (group.name, n_bad, rejected + n_spacers)
        n_streams += len(group.cases)
    print("%s: %d streams compared (%d accepted by zlib), %.1f s" % (family, n_streams, n_accept, time.time() - t0))
    assert not bad, "%d of %d stream(s) decoded differently from zlib:\n%s" % (len(bad), n_streams, "\n".join(bad))

