import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
ALGS = ("chameleon", "cheetah", "lion")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def splitmix_bytes(n, seed):
    """SURVEY.md §8c footnote 1 (vectorised)."""
    M = np.uint64(0xFFFFFFFFFFFFFFFF)
    i = np.arange(1, (n + 7) // 8 + 1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = (np.uint64(seed) + i * np.uint64(0x9E3779B97F4A7C15)) & M
        z = x
        z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & M
        z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & M
        z = z ^ (z >> np.uint64(31))
    return z.view(np.uint8)[:n].copy()


@pytest.fixture(scope="session")
def golden():
    return json.load(open(os.path.join(GOLDEN_DIR, "golden.json")))


@pytest.fixture(scope="session")
def dickens200k():
    return np.fromfile(os.path.join(GOLDEN_DIR, "dickens_200k.bin"), dtype=np.uint8)


@pytest.fixture(scope="session")
def golden_inputs(dickens200k):
    d = dickens200k
    cases = {
        "kat": np.frombuffer(b"test" * 31 + b"t", dtype=np.uint8),
        "dickens_65539": d[:65539],
        "zeros_1m": np.zeros(1 << 20, dtype=np.uint8),
        "splitmix_1m_seed1": splitmix_bytes(1 << 20, 1),
        "mixed_280004": np.concatenate([d[:100000], splitmix_bytes(50001, 7), np.zeros(30000, np.uint8), d[100000:200003]]),
        # stands in for the whole 10 MB file, whose digests stay in golden.json for test_published_dickens_ratios
        "dickens_sample_256k": np.fromfile(os.path.join(GOLDEN_DIR, "dickens_sample_256k.bin"), dtype=np.uint8),
    }
    return cases


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def payload(kind, n, seed=0):
    """Small seeded test payloads: text-like, random, zeros, low-entropy, mixed."""
    rng = np.random.default_rng(seed * 7919 + n)
    if kind == "zeros":
        return np.zeros(n, np.uint8)
    if kind == "random":
        return rng.integers(0, 256, n, dtype=np.uint8)
    if kind == "low":
        return rng.integers(0, 4, n, dtype=np.uint8)
    if kind == "text":
        d = np.fromfile(os.path.join(GOLDEN_DIR, "dickens_200k.bin"), dtype=np.uint8)
        off = int(rng.integers(0, max(1, d.size - n))) if n < d.size else 0
        out = np.resize(d[off:], n) if n > d.size - off else d[off:off + n]
        return out.copy()
    if kind == "mixed":
        parts, left = [], n
        while left > 0:
            k = int(min(left, rng.integers(1, 4000)))
            parts.append(payload(["text", "random", "zeros", "low"][int(rng.integers(0, 4))], k, seed + len(parts) + 1))
            left -= k
        return np.concatenate(parts)[:n] if parts else np.zeros(0, np.uint8)
    raise ValueError(kind)
