"""GPU DEFLATE vs the CPU model (tests/model, the kernel's parameters): every stream of `python tools/check_model.py
[MiB]` MiB of corpus text, CDC-chunked with the text dictionary, must equal the model's byte for byte (same candidate
sets, same parse, same Huffman codes).  Prints the first differences in stream terms.  TEST INFRASTRUCTURE;
tests/test_gpu_deflate_exact.py runs the same comparison on many more inputs."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hmse_b200  # noqa: E402
from oracle import corpus  # noqa: E402
from tests.model import exact  # noqa: E402
from tests.model.inflate_tokens import first_difference  # noqa: E402


def main():
    mib = int(sys.argv[1]) if len(sys.argv) > 1 else 4
    data = corpus.generate(mib << 20)
    zd = corpus.zdict()
    ctx = hmse_b200.default_context(0)
    cuts = hmse_b200.chunk(data, hmse_b200.CDCConfig(), ctx=ctx)
    blob, offs = hmse_b200.compress(data, cuts, None, zd, ctx=ctx)
    offs = np.asarray(offs).astype(np.int64)
    case = exact.Case("corpus", data, cuts, zd)
    want = case.expected(exact.Model())
    bad = 0
    for k, w in enumerate(want):
        g = blob[offs[k]:offs[k + 1]].tobytes()
        if g != w:
            bad += 1
            if bad <= 5:
                n = len(case.chunk(k))
                print("chunk", k, "len", n, exact.size_class(n), "gpu", len(g), "model", len(w), "-", first_difference(g, w))
    print("chunks", len(want), "differing streams", bad, "gpu bytes", int(offs[-1]), "model bytes", sum(len(w) for w in want))


if __name__ == "__main__":
    main()
