"""Regenerates tests/golden/* from the Silesia corpus file `dickens` (10,192,446 bytes):

    python tests/golden/make_golden.py path/to/dickens

The expected outputs are produced by the oracle (oracle/density_oracle.c), which is itself pinned on the reference's
known-answer vectors (the reference's src/lib.rs:19,28,50,72). The reference is Rust and this project does not build it,
so these fixtures are "oracle outputs cross-checked against the reference's published facts":
  * the three KATs (exact bytes),
  * dickens compressed sizes 5,827,114 / 5,480,246 / 5,183,816 <=> ratios 1.749x/1.860x/1.966x (benchmark.log:17,22,27),
  * the independently derived digests listed in SURVEY.md §8c.
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
import oracle  # noqa: E402

SAMPLE_PIECES, SAMPLE_PIECE_BYTES = 16, 16384


def splitmix_bytes(n, seed):
    out = np.empty((n + 7) // 8, dtype=np.uint64)
    x = seed
    M = (1 << 64) - 1
    for i in range(out.size):
        x = (x + 0x9E3779B97F4A7C15) & M
        z = x
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
        out[i] = z ^ (z >> 31)
    return out.view(np.uint8)[:n].copy()


def dickens_sample(d):
    """16 KiB pieces at 16 evenly spaced offsets of the whole file: the full file is too large to keep in the tree."""
    step = d.size // SAMPLE_PIECES
    return np.concatenate([d[k * step:k * step + SAMPLE_PIECE_BYTES] for k in range(SAMPLE_PIECES)])


def main(path):
    d = np.frombuffer(open(path, "rb").read(), dtype=np.uint8)
    d[:200003].tofile(os.path.join(HERE, "dickens_200k.bin"))
    sample = dickens_sample(d)
    sample.tofile(os.path.join(HERE, "dickens_sample_256k.bin"))
    cases = {
        "kat": np.frombuffer(b"test" * 31 + b"t", dtype=np.uint8),
        "dickens_65539": d[:65539],
        "zeros_1m": np.zeros(1 << 20, dtype=np.uint8),
        "splitmix_1m_seed1": splitmix_bytes(1 << 20, 1),
        "mixed_280004": np.concatenate([d[:100000], splitmix_bytes(50001, 7), np.zeros(30000, np.uint8), d[100000:200003]]),
        "dickens_full": d,
        "dickens_sample_256k": sample,
    }
    gold = {}
    for name, data in cases.items():
        entry = {"input_len": int(data.size), "input_sha256": hashlib.sha256(data.tobytes()).hexdigest(), "alg": {}}
        for alg in ("chameleon", "cheetah", "lion"):
            enc, copied = oracle.encode(alg, data, return_copied=True)
            dec = oracle.decode(alg, enc, data.size)
            assert dec.size == data.size and (dec == data).all()
            entry["alg"][alg] = {"size": int(enc.size), "sha256": hashlib.sha256(enc.tobytes()).hexdigest(), "copied_blocks": int(copied)}
            if name == "kat":
                entry["alg"][alg]["bytes"] = enc.tolist()
        gold[name] = entry
        print(name, {a: (v["size"], v["sha256"][:32], v["copied_blocks"]) for a, v in entry["alg"].items()})
    json.dump(gold, open(os.path.join(HERE, "golden.json"), "w"), indent=1)


if __name__ == "__main__":
    main(sys.argv[1])
