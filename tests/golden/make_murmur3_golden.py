"""Regenerates tests/golden/murmur3_sklearn.json (run from the repo root: `python tests/golden/make_murmur3_golden.py`;
needs scikit-learn).  scikit-learn ships its own C++ copy of Appleby's MurmurHash3_x86_32
(sklearn.utils.murmurhash3_32, written by other people than the oracle's); its answers are stored here so that
tests/test_oracle_kat.py pins the oracle's hash and MinHash against an independent implementation whether or not
scikit-learn is installed.  Inputs: random keys of every length 0..40 with random seeds, and the MinHash minima of
four chunks of the first 6000 bytes of the seed-42 corpus (one of them 3 bytes long: no shingle)."""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import corpus  # noqa: E402

MINHASH_CUTS = [1000, 1003, 4096, 6000]
MINHASH_PERMS = [0, 17, 127]


def vectors():
    from sklearn.utils import murmurhash3_32
    rng = np.random.default_rng(2024)
    hashes = []
    for n in range(0, 41):
        for _ in range(8):
            key = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
            seed = int(rng.integers(0, 1 << 32))
            hashes.append([key.hex(), seed, int(murmurhash3_32(key, seed=seed, positive=True))])
    data = corpus.generate(MINHASH_CUTS[-1])
    raw = data.tobytes()
    mins, lo = [], 0
    for j, hi in enumerate(MINHASH_CUTS):
        shingles = {raw[i:i + 4] for i in range(lo, hi - 3)}
        for p in MINHASH_PERMS:
            mins.append([j, p, min((int(murmurhash3_32(s, seed=p + 1, positive=True)) for s in shingles), default=0xFFFFFFFF)])
        lo = hi
    return {"hashes": hashes, "minhash": {"input_sha256": hashlib.sha256(raw).hexdigest(), "cuts": MINHASH_CUTS, "mins": mins}}


def main():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "murmur3_sklearn.json"), "w") as f:
        json.dump(vectors(), f, indent=0)
    print("wrote murmur3_sklearn.json")


if __name__ == "__main__":
    main()
