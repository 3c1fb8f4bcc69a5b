"""Parity of the CUDA path against the oracle, through the C ABI (needs a B200: pytest -m gpu).

Bit-exact bar: every byte of every encoded stream equals the oracle's; every decode equals the original."""
import os

import numpy as np
import pytest

import oracle
from conftest import ALGS, payload, sha256, splitmix_bytes

pytestmark = pytest.mark.gpu

TEST_DATA = b"test" * 31 + b"t"


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    return torch


@pytest.fixture(scope="module")
def codecs(torch_cuda):
    import density_b200
    density_b200.load()  # raises if the CUDA extension is missing
    return density_b200.CODECS


def gpu_encode(C, data):
    out = np.zeros(max(1, C.safe_encode_buffer_size(data.size)), dtype=np.uint8)
    n = C.encode(data, out)
    return out[:n]


def gpu_decode(C, enc, n):
    out = np.zeros(max(1, n), dtype=np.uint8)
    m = C.decode(enc, out)
    return out[:m]


@pytest.mark.parametrize("alg", ALGS)
def test_reference_kats_through_c_abi(codecs, alg, golden):
    C = codecs[alg]
    data = np.frombuffer(TEST_DATA, dtype=np.uint8)
    out = np.zeros(len(TEST_DATA), dtype=np.uint8)  # same undersized-but-sufficient buffer as lib.rs:24
    n = C.encode(data, out)
    assert out[:n].tolist() == golden["kat"]["alg"][alg]["bytes"]
    assert gpu_decode(C, out[:n], len(TEST_DATA)).tobytes() == TEST_DATA


@pytest.mark.parametrize("alg", ALGS)
def test_golden_fixtures_encode_decode(codecs, alg, golden, golden_inputs):
    C = codecs[alg]
    for name, data in golden_inputs.items():
        enc = gpu_encode(C, data)
        e = golden[name]["alg"][alg]
        assert (enc.size, sha256(enc)) == (e["size"], e["sha256"]), (alg, name)
        dec = gpu_decode(C, enc, data.size)
        assert dec.size == data.size and (dec == data).all(), (alg, name)


@pytest.mark.parametrize("alg", ALGS)
@pytest.mark.parametrize("kind", ["text", "random", "zeros", "low", "mixed"])
def test_tail_and_copy_mode_sweep_vs_oracle(codecs, alg, kind):
    C = codecs[alg]
    for n in [1, 2, 3, 4, 5, 7, 8, 15, 16, 17, 63, 64, 65, 127, 128, 129, 255, 256, 257, 260, 511, 512, 513, 1000, 2999,
              16383, 16384, 16385, 16387, 70001]:
        data = payload(kind, n, seed=n)
        want = oracle.encode(alg, data)
        got = gpu_encode(C, data)
        assert got.size == want.size and (got == want).all(), (alg, kind, n)
        dec = gpu_decode(C, got, n)
        assert dec.size == n and (dec == data).all(), (alg, kind, n)


@pytest.mark.parametrize("alg", ALGS)
def test_empty_input(codecs, alg):
    C = codecs[alg]
    assert C.encode(np.zeros(0, np.uint8), np.zeros(8, np.uint8)) == 0
    assert C.decode(np.zeros(0, np.uint8), np.zeros(8, np.uint8)) == 0


@pytest.mark.parametrize("path", [0, 1, 2, 3])
@pytest.mark.parametrize("nbytes", [300, 16 * 1024, 16 * 1024 + 4, 1 << 20, (1 << 22) + 777, 9 * (1 << 20) + 2])
def test_chameleon_every_device_path_on_text(torch_cuda, codecs, path, nbytes):
    """path 0 auto, 1 parallel fast path only, 2 in-order protected walk, 3 scalar kernel: all bit-identical on quiet text."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    if path == 3 and nbytes > (1 << 22) + 777:
        pytest.skip("scalar kernel is slow")
    data = synth.synth_text(nbytes).numpy()
    want = oracle.encode("chameleon", data)
    d_in = torch.from_numpy(data).cuda()
    d_out = torch.zeros(codecs["chameleon"].safe_encode_buffer_size(nbytes) + 64, dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.encode_device("chameleon", d_in, d_out, d_sz, path=path)
    torch.cuda.synchronize()
    n = int(d_sz.item())
    got = d_out[:n].cpu().numpy()
    assert n == want.size and (got == want).all()


@pytest.mark.parametrize("kind", ["random", "mixed", "low", "zeros"])
@pytest.mark.parametrize("nbytes", [70001, 1 << 20, 3 * (1 << 20) + 5])
def test_chameleon_non_quiet_inputs_fall_back_exactly(codecs, kind, nbytes):
    C = codecs["chameleon"]
    data = payload(kind, nbytes, seed=3)
    want = oracle.encode("chameleon", data)
    got = gpu_encode(C, data)
    assert got.size == want.size and (got == want).all()


def _same_bucket_pair():
    M = 0x9D6EF916
    seen = {}
    q = 0x12345678
    while True:
        q = (q * 1103515245 + 12345) & 0xFFFFFFFF
        h = ((q * M) & 0xFFFFFFFF) >> 16
        if h in seen and seen[h] != q:
            return seen[h], q
        seen[h] = q



@pytest.mark.gpu
@pytest.mark.parametrize("impl", [6, 1])
def test_chameleon_runs_of_equal_quads_and_mailbox_overflow(torch_cuda, codecs, impl):
    """Round-2 flag pass (write / verify / mailbox): runs of equal quads of every length up to several tiles (one mailbox entry per run:
    the run is dropped at deposit time), runs cut by a different quad of the same bucket, 5 - 40 quads of one bucket that are NOT a run
    (main mailbox -> overflow mailboxes -> in-order replay of the tile), all inside text so that most blocks stay compressible; the
    round-1 kernel must agree (impl 1)."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    rng = np.random.default_rng(5)
    q1, q2 = _same_bucket_pair()
    text = synth.synth_text(6 << 20).numpy().view(np.uint32).copy()
    pieces, pos = [], 0
    lens = [1, 2, 3, 5, 31, 32, 33, 64, 255, 256, 257, 1000, 4095, 4096, 4097, 9000]
    vals = [0, 0xFFFFFFFF, 0x20202020, q1, q2, 0x80000000, 1]
    k = 0
    while pos + 20000 < text.size:
        step = int(rng.integers(3000, 20000))
        pieces.append(text[pos:pos + step]); pos += step
        L = lens[k % len(lens)]; v = vals[k % len(vals)]
        if k % 3 == 0:
            pieces.append(np.full(L, v, dtype=np.uint32))                                   # a plain run
        elif k % 3 == 1:
            run = np.full(L, q1, dtype=np.uint32); run[L // 2] = q2                          # a run cut by a quad of the same bucket
            pieces.append(run)
        else:
            m = 5 + (k % 36)                                                                 # m dirty members of one bucket, no two adjacent equal
            burst = np.empty(2 * m, dtype=np.uint32); burst[0::2] = q1 if (k & 1) else q2; burst[1::2] = text[pos:pos + m]
            burst[0::4] = q2 if (k & 1) else q1
            pieces.append(burst)
        k += 1
    data = np.concatenate(pieces).view(np.uint8)[:-1]
    want = oracle.encode("chameleon", data)
    lib = density_b200.load()
    lib.density_b200_test_set_flag_impl(impl)
    try:
        for path in (0, 1):
            d_in = torch.from_numpy(data.copy()).cuda()
            d_out = torch.zeros(codecs["chameleon"].safe_encode_buffer_size(data.size) + 64, dtype=torch.uint8, device="cuda")
            d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
            density_b200.encode_device("chameleon", d_in, d_out, d_sz, path=path)
            torch.cuda.synchronize()
            n = int(d_sz.item())
            if path == 1 and n == 0:
                continue          # path 1 = parallel only: gives up (size 0) when the copy map does not settle; path 0 must still be exact
            assert n == want.size and (d_out[:n].cpu().numpy() == want).all(), (impl, path)
        # and back through the decoder (both decode pass kernels)
        for dimpl in (7, 1):
            lib.density_b200_test_set_decode_impl(dimpl)
            d_enc = torch.from_numpy(want.copy()).cuda()
            d_dec = torch.zeros(data.size + 64, dtype=torch.uint8, device="cuda")
            density_b200.decode_device("chameleon", d_enc, want.size, d_dec, d_sz, path=0)
            torch.cuda.synchronize()
            assert int(d_sz.item()) == data.size and (d_dec[:data.size].cpu().numpy() == data).all(), dimpl
    finally:
        lib.density_b200_test_set_flag_impl(6)
        lib.density_b200_test_set_decode_impl(7)


@pytest.mark.parametrize("path", [0, 1, 2])
def test_chameleon_adversarial_same_bucket_alternation(torch_cuda, codecs, path):
    """Thousands of interleaving quads in ONE hash bucket per tile (class-list overflow -> sequential in-tile fallback),
    padded with zero runs so that every block stays compressible and the stream stays on the parallel path."""
    torch = torch_cuda
    import density_b200
    q1, q2 = _same_bucket_pair()
    block = np.array([q1, q2] * 20 + [0] * 24, dtype=np.uint32)
    data = np.tile(block, 3000).view(np.uint8)[: 3000 * 256 - 3]
    want, copied = oracle.encode("chameleon", data, return_copied=True)
    assert copied == 0
    d_in = torch.from_numpy(data.copy()).cuda()
    d_out = torch.zeros(codecs["chameleon"].safe_encode_buffer_size(data.size) + 64, dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.encode_device("chameleon", d_in, d_out, d_sz, path=path)
    torch.cuda.synchronize()
    n = int(d_sz.item())
    assert n == want.size and (d_out[:n].cpu().numpy() == want).all()
    if path == 1:
        assert density_b200.load().density_b200_last_encode_was_fast() == 1


def test_chameleon_many_runs_64mib_text(torch_cuda, codecs):
    """148 runs of >=16 tiles each: exercises the carry-in / unresolved machinery across every SM."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    n = 64 * (1 << 20) + 1234
    d_in = synth.synth_text(n, device="cuda")
    data = d_in.cpu().numpy()
    want = oracle.encode("chameleon", data)
    d_out = torch.zeros(codecs["chameleon"].safe_encode_buffer_size(n), dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.encode_device("chameleon", d_in, d_out, d_sz, path=1)
    torch.cuda.synchronize()
    got = d_out[:int(d_sz.item())].cpu().numpy()
    assert got.size == want.size and (got == want).all()
    assert density_b200.load().density_b200_last_encode_was_fast() == 1


def test_chameleon_full_size_1gib_text_bit_exact(torch_cuda, codecs):
    """BASELINE.json configs[1] at full size: bit-exact against the oracle, plus the size-independent checks
    (round trip of a prefix through the decoder; determinism across two runs)."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    n = 1 << 30
    d_in = synth.synth_text(n, device="cuda")
    d_out = torch.zeros(codecs["chameleon"].safe_encode_buffer_size(n), dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.encode_device("chameleon", d_in, d_out, d_sz)
    torch.cuda.synchronize()
    m = int(d_sz.item())
    assert density_b200.load().density_b200_last_encode_was_fast() == 1
    got = d_out[:m].cpu().numpy()
    want = oracle.encode("chameleon", d_in.cpu().numpy())
    assert m == want.size
    assert (got == want).all()
    # determinism
    d_out2 = torch.zeros_like(d_out)
    density_b200.encode_device("chameleon", d_in, d_out2, d_sz)
    torch.cuda.synchronize()
    assert int(d_sz.item()) == m and torch.equal(d_out[:m], d_out2[:m])


def test_chameleon_beyond_4gib_prefix_and_round_trip(torch_cuda, codecs):
    """5 GiB of text in one call (byte offsets past 2^32, the per-GPU shard scale of SURVEY.md §8d config 5). Size-independent checks:
    the stream of a prefix is a prefix of the stream (codec.rs:72-80 walks the blocks in order; a 64 MiB prefix is compared with the
    oracle), the stream decodes back to the input on the device, and the output size obeys codec.rs:18-21."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    C = codecs["chameleon"]
    n = 5 * (1 << 30) + 256 * 3 + 1
    if torch.cuda.mem_get_info()[0] < 24 * (1 << 30):
        pytest.skip("needs 24 GiB of free device memory")
    d_in = torch.empty(n, dtype=torch.uint8, device="cuda")
    for off in range(0, n, 1 << 30):                       # page-aligned pieces of the same counter-based text
        k = min(1 << 30, n - off)
        d_in[off:off + k] = synth.synth_text(k, device="cuda", first_page=off // synth.PAGE)
    d_out = torch.empty(C.safe_encode_buffer_size(n), dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.encode_device("chameleon", d_in, d_out, d_sz)
    torch.cuda.synchronize()
    m = int(d_sz.item())
    assert 0 < m <= C.safe_encode_buffer_size(n)
    npre = 64 << 20
    want = oracle.encode("chameleon", d_in[:npre].cpu().numpy())
    assert (d_out[:want.size].cpu().numpy() == want).all()
    d_dec = torch.empty(n, dtype=torch.uint8, device="cuda")
    density_b200.decode_device("chameleon", d_out, m, d_dec, d_sz)
    torch.cuda.synchronize()
    assert int(d_sz.item()) == n and torch.equal(d_dec, d_in)


def test_chameleon_encode_chained_copy_mode_episodes(torch_cuda, codecs):
    """The same incompressible blob 14 times in 64 MiB of text: episode k sees what episode k-1 left in the dictionary (the text never
    touches those buckets), so the copy map settles one episode per fixed-point round. The reference-facing entry point keeps
    iterating from the host instead of dropping to the in-order walk; the result is the oracle's stream either way."""
    torch = torch_cuda
    import ctypes
    import density_b200
    from density_b200 import synth
    n = 64 * (1 << 20) + 100
    data = synth.synth_text(n).numpy().copy()
    blob = synth.random_bytes(65536, 99).numpy()
    for k in range(14):
        off = (2 + 4 * k) * (1 << 20) + 256 * k
        data[off:off + blob.size] = blob
    want, copied = oracle.encode("chameleon", data, return_copied=True)
    assert copied > 0
    d_in = torch.from_numpy(data).cuda()
    d_out = torch.zeros(codecs["chameleon"].safe_encode_buffer_size(n), dtype=torch.uint8, device="cuda")
    m = codecs["chameleon"].encode(d_in, d_out)            # chameleon_encode(): device pointers, synchronous
    assert m == want.size and (d_out[:m].cpu().numpy() == want).all()
    st = (ctypes.c_uint64 * 6)()
    assert density_b200.load().density_b200_encode_status(st) == 0
    assert st[1] == 1 and st[4] == 1, "copy map should have settled by iteration, not by the in-order walk"
    # the stream-ordered auto path (fixed round budget, in-order walk as the fallback) gives the same bytes
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    d_out.zero_()
    density_b200.encode_device("chameleon", d_in, d_out, d_sz, path=0)
    torch.cuda.synchronize()
    assert int(d_sz.item()) == want.size and (d_out[:want.size].cpu().numpy() == want).all()


@pytest.mark.parametrize("alg", ["cheetah", "lion"])
@pytest.mark.parametrize("nbytes", [33 * (1 << 20) + 66, (1 << 20) + 5])
def test_cheetah_lion_blocking_iteration_resumes(torch_cuda, codecs, alg, nbytes):
    """Path 4 (what the synchronous reference symbols use): when the copy map has not settled after the enqueued stages the host reads
    the verdict and resumes the iteration instead of leaving the stream to the in-order kernel. The test hook cuts every stage to one
    round so that the resume path is exercised on ordinary text; the in-order kernel would need seconds for the larger input."""
    import time
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    data = synth.synth_text(nbytes).numpy()
    want = oracle.encode(alg, data)
    d_in = torch.from_numpy(data.copy()).cuda()
    d_out = torch.zeros(codecs[alg].safe_encode_buffer_size(nbytes) + 64, dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.encode_device(alg, d_in, d_out, d_sz, path=4)          # warm (workspace allocation)
    torch.cuda.synchronize()
    density_b200.load().density_b200_test_set_stage_rounds(1)
    try:
        d_out.zero_(); d_sz.zero_()
        t0 = time.perf_counter()
        density_b200.encode_device(alg, d_in, d_out, d_sz, path=4)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    finally:
        density_b200.load().density_b200_test_set_stage_rounds(7)
    n = int(d_sz.item())
    assert n == want.size and (d_out[:n].cpu().numpy() == want).all()
    if nbytes > (1 << 25):
        assert dt < 1.0, f"{dt:.2f} s: the in-order kernel produced this, not the resumed iteration"


@pytest.mark.parametrize("alg", ALGS)
def test_device_pointers_through_reference_symbols(torch_cuda, codecs, alg):
    torch = torch_cuda
    C = codecs[alg]
    data = payload("text", 50000, 5)
    d_in = torch.from_numpy(data).cuda()
    d_out = torch.zeros(C.safe_encode_buffer_size(data.size), dtype=torch.uint8, device="cuda")
    n = C.encode(d_in, d_out)
    want = oracle.encode(alg, data)
    assert n == want.size and (d_out[:n].cpu().numpy() == want).all()
    d_dec = torch.zeros(data.size, dtype=torch.uint8, device="cuda")
    m = C.decode(d_out[:n].clone(), d_dec)
    assert m == data.size and (d_dec.cpu().numpy() == data).all()


@pytest.mark.parametrize("alg", ALGS)
def test_error_behaviour_returns_zero_never_aborts(codecs, alg):
    from density_b200 import DecodeError, EncodeError
    C = codecs[alg]
    data = splitmix_bytes(4096, 11)
    with pytest.raises(EncodeError):   # output too small for incompressible data: reference would panic (write_buffer.rs:19)
        C.encode(data, np.zeros(1000, dtype=np.uint8))
    enc = gpu_encode(C, payload("text", 4096, 2))
    with pytest.raises(DecodeError):   # output too small
        C.decode(enc, np.zeros(100, dtype=np.uint8))
    with pytest.raises(DecodeError):   # truncated inside a signature
        C.decode(enc[:3], np.zeros(4096, dtype=np.uint8))


def test_decode_oracle_streams_and_vice_versa(codecs):
    """Streams are interchangeable with the reference's in both directions."""
    for alg in ALGS:
        C = codecs[alg]
        data = payload("mixed", 200000, 9)
        enc_cpu = oracle.encode(alg, data)
        assert (gpu_decode(C, enc_cpu, data.size) == data).all()
        enc_gpu = gpu_encode(C, data)
        assert (oracle.decode(alg, enc_gpu, data.size) == data).all()


def test_sharded_stream_equals_single_call(torch_cuda, codecs):
    """SURVEY §8e on one GPU: cut one stream into 3 shards, run phase 1 on each, fold the exported tables left to
    right, run phase 2 with the carried-in dictionary; the concatenation must equal the oracle's single-call output."""
    torch = torch_cuda
    import ctypes
    import density_b200
    from density_b200 import sharded, synth
    L = density_b200.load()
    n = 3 * (1 << 21) + 515
    data = synth.synth_text(n).numpy()
    want = oracle.encode("chameleon", data)
    cuts = [0, 1 << 21, (1 << 21) + (1 << 20) + 256 * 7, n]
    encs, tables, ins = [], [], []
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for r in range(3):
        d_in = torch.from_numpy(data[cuts[r]:cuts[r + 1]].copy()).cuda()
        t = torch.empty(65536, dtype=torch.int32, device="cuda")
        e = sharded.ShardedChameleonEncoder()
        rc = L.density_b200_shard_phase1(e._h, d_in.data_ptr(), d_in.numel(), int(r == 2), t.data_ptr(), stream)
        assert rc == 0, density_b200._lib.last_error()
        encs.append(e); tables.append(t); ins.append(d_in)
    gathered = torch.stack(tables)
    pieces = []
    for r in range(3):
        carry = sharded.fold_tables(gathered, r) if r > 0 else None
        d_out = torch.zeros(codecs["chameleon"].safe_encode_buffer_size(ins[r].numel()) + 64, dtype=torch.uint8, device="cuda")
        d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
        d_fl = torch.zeros(1, dtype=torch.int32, device="cuda")
        rc = L.density_b200_shard_phase2(encs[r]._h, carry.data_ptr() if carry is not None else None, d_out.data_ptr(),
                                         d_out.numel(), d_sz.data_ptr(), d_fl.data_ptr(), stream)
        assert rc == 0, density_b200._lib.last_error()
        torch.cuda.synchronize()
        assert int(d_fl.item()) == 0
        pieces.append(d_out[:int(d_sz.item())].cpu().numpy())
    got = np.concatenate(pieces)
    assert got.size == want.size and (got == want).all()


@pytest.mark.parametrize("kind", ["text", "mixed"])
def test_chameleon_host_pipelined_path_bit_exact(torch_cuda, codecs, kind):
    """>= 96 MiB host buffers take the PCIe-pipelined path (64 MiB chunks as shards of one stream); a non-quiet input
    makes it fall back to the whole-buffer protection-aware path. Both must equal the oracle."""
    from density_b200 import synth
    n = 160 * (1 << 20) + 12345
    data = (synth.synth_text(n) if kind == "text" else synth.synth_mixed(n)).numpy()
    want = oracle.encode("chameleon", data)
    got = gpu_encode(codecs["chameleon"], data)
    assert got.size == want.size and (got == want).all()


@pytest.mark.gpu
def test_chameleon_host_pipelined_path_tiny_last_chunk(torch_cuda, codecs):
    """The pipelined host path cuts the input into 64 MiB chunks: a 5-byte last chunk (no whole quad) must come out like the
    oracle's tail, from pageable host buffers (staged through the pinned ring)."""
    from density_b200 import synth
    n = 128 * (1 << 20) + 5
    data = synth.synth_text(n).numpy()
    want = oracle.encode("chameleon", data)
    got = gpu_encode(codecs["chameleon"], data)
    assert got.size == want.size and (got == want).all()


@pytest.mark.parametrize("path", [0, 1, 3])
@pytest.mark.parametrize("nbytes", [5, 263, 264, 300, 4096, 16 * 1024 + 4, 70001, 1 << 20, (1 << 22) + 777, 24 * (1 << 20) + 3])
def test_chameleon_decode_paths_on_text(torch_cuda, codecs, path, nbytes):
    """path 0 auto, 1 parallel decoder only (boundary chase + tile protocol + in-order tail), 3 in-order kernel: identical."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    if path == 3 and nbytes > (1 << 22) + 777:
        pytest.skip("in-order kernel is slow")
    data = synth.synth_text(nbytes).numpy()
    enc = oracle.encode("chameleon", data)          # a stream produced by the reference algorithm on the CPU
    d_enc = torch.from_numpy(enc).cuda()
    d_out = torch.zeros(nbytes + 64, dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.decode_device("chameleon", d_enc, enc.size, d_out, d_sz, path=path)
    torch.cuda.synchronize()
    assert int(d_sz.item()) == nbytes
    assert (d_out[:nbytes].cpu().numpy() == data).all()


@pytest.mark.parametrize("path", [0, 1])
@pytest.mark.parametrize("kind,nbytes", [("random", 3 * (1 << 20) + 5), ("mixed", 3 * (1 << 20) + 5), ("low", 3 * (1 << 20) + 5), ("zeros", 3 * (1 << 20) + 5),
                                         ("random", 70001), ("mixed", 280004), ("random", 256 * 40 + 263), ("random", 256 * 40 + 264),
                                         ("smixed", 40 * (1 << 20) + 3), ("bursts", 24 * (1 << 20) + 777)])
def test_chameleon_decode_copy_mode_streams(torch_cuda, codecs, path, kind, nbytes):
    """Streams with copy-mode blocks (codec.rs:89-92): the candidate boundary walks are void, `dec_seq_walk` redoes the boundaries in
    order with the exact automaton and the parallel dictionary passes run on its block list. path 1 = parallel decoder only (no
    in-order fallback), so this is the parallel path being checked; the streams come from the oracle."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    if kind == "bursts":      # text with a few incompressible bursts: most chunks are jumped over, the ones around the bursts are walked
        data = synth.synth_text(nbytes).numpy().copy()
        for off, ln in ((1 << 20, 65536), (5 * (1 << 20) + 300, 1500), (17 * (1 << 20) + 2, 300000), (nbytes - 3000, 3000)):
            data[off:off + ln] = synth.random_bytes(ln, 99).numpy()
    else:
        data = synth.synth_mixed(nbytes).numpy() if kind == "smixed" else payload(kind, nbytes, seed=5)
    enc, copied = oracle.encode("chameleon", data, return_copied=True)
    if kind in ("random", "mixed", "smixed", "bursts"):
        assert copied > 0
    d_enc = torch.from_numpy(enc.copy()).cuda()
    d_out = torch.zeros(nbytes + 64, dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.decode_device("chameleon", d_enc, enc.size, d_out, d_sz, path=path)
    torch.cuda.synchronize()
    if path == 1 and int(d_sz.item()) == 0 and kind in ("low", "zeros"):
        pytest.skip("pathological tile (thousands of readers of one freshly written bucket): path 0 falls back to the in-order kernel")
    assert int(d_sz.item()) == nbytes
    assert (d_out[:nbytes].cpu().numpy() == data).all()
    # host-pointer entry point (the reference symbol) on the same stream
    if nbytes <= 3 * (1 << 20) + 5:
        dec = gpu_decode(codecs["chameleon"], enc, data.size)
        assert dec.size == data.size and (dec == data).all()


def test_chameleon_decode_adversarial_same_bucket(torch_cuda, codecs):
    """writers (plain quads) of ONE bucket interleaved with readers of that bucket inside every tile."""
    q1, q2 = _same_bucket_pair()
    block = np.array([q1, q1, q2, q2, q2, q1] * 6 + [0] * 28, dtype=np.uint32)
    data = np.tile(block, 2500).view(np.uint8)[: 2500 * 256 - 1]
    enc, copied = oracle.encode("chameleon", data, return_copied=True)
    assert copied == 0
    dec = gpu_decode(codecs["chameleon"], enc, data.size)
    assert dec.size == data.size and (dec == data).all()


@pytest.mark.parametrize("alg", ["cheetah", "lion"])
@pytest.mark.parametrize("path", [0, 1, 3])
@pytest.mark.parametrize("kind,nbytes", [("text", 300), ("text", 4096 + 3), ("text", 70001), ("text", (1 << 20) + 5), ("text", 6 * (1 << 20) + 2),
                                         ("mixed", 3 * (1 << 20) + 1), ("random", 1 << 20), ("zeros", 1 << 20), ("low", 500000),
                                         ("dickens", 200000), ("text", 33 * (1 << 20) + 66)])
def test_cheetah_lion_encode_paths(torch_cuda, codecs, alg, path, kind, nbytes):
    """path 0 auto (run-parallel encoder, in-order kernel if the copy map does not settle), 1 run-parallel only, 3 in-order kernel.

    cheetah.rs:121-150 / lion.rs:209-271 through codec.rs:34-80. With path 1 an output size of 0 means "copy map not settled within the
    round budget" (the caller must then use path 0): tolerated only where the copy-mode automaton is busy all over the input."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    if path == 3 and nbytes > (1 << 20) + 5:
        pytest.skip("in-order kernel is slow")
    if kind == "dickens":
        data = np.fromfile(os.path.join(os.path.dirname(__file__), "golden", "dickens_200k.bin"), np.uint8)[:nbytes]
    else:
        data = synth.synth_text(nbytes).numpy() if kind == "text" else (synth.synth_mixed(nbytes).numpy() if kind == "mixed" else payload(kind, nbytes, 7))
    want = oracle.encode(alg, data)
    d_in = torch.from_numpy(data.copy()).cuda()
    d_out = torch.zeros(codecs[alg].safe_encode_buffer_size(nbytes) + 64, dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.encode_device(alg, d_in, d_out, d_sz, path=path)
    torch.cuda.synchronize()
    n = int(d_sz.item())
    if path == 1 and n == 0 and kind in ("mixed", "dickens"):
        pytest.skip("copy map not settled by the parallel rounds (path 0 falls back to the in-order kernel)")
    assert n == want.size and (d_out[:n].cpu().numpy() == want).all()


def _device_mixed(torch, synth, n):
    """n bytes of the synthetic mixed text/binary corpus on the device, generated in 1 GiB pieces (region-aligned, so the pieces
    concatenate to the same bytes as one call)."""
    d = torch.empty(n, dtype=torch.uint8, device="cuda")
    step = 1 << 30
    for off in range(0, n, step):
        k = min(step, n - off)
        d[off:off + k] = synth.synth_mixed(k, device="cuda", first_region=off // synth.REGION)
    return d


def test_cheetah_full_size_1gib_text_bit_exact(torch_cuda, codecs):
    """BASELINE.json configs[2] (encode half) at full size: Cheetah encode of the 1 GiB synthetic text, every byte against the oracle
    (cheetah.rs:121-150 through codec.rs:34-80)."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    n = 1 << 30
    d_in = synth.synth_text(n, device="cuda")
    d_out = torch.zeros(codecs["cheetah"].safe_encode_buffer_size(n), dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.encode_device("cheetah", d_in, d_out, d_sz, path=1)     # run-parallel encoder only: no in-order fallback
    torch.cuda.synchronize()
    m = int(d_sz.item())
    want = oracle.encode("cheetah", d_in.cpu().numpy())
    assert m == want.size
    assert (d_out[:m].cpu().numpy() == want).all()


def test_lion_full_size_4gib_mixed_bit_exact(torch_cuda, codecs):
    """BASELINE.json configs[3] at full size: Lion encode of the 4 GiB mixed text/binary buffer (2^32 bytes: quad and byte offsets
    cross 32 bits), every byte against the oracle (lion.rs:209-271 through codec.rs:34-80)."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    n = 1 << 32
    if torch.cuda.mem_get_info()[0] < 40 * (1 << 30):
        pytest.skip("needs 40 GiB of free device memory")
    d_in = _device_mixed(torch, synth, n)
    C = codecs["lion"]
    d_out = torch.empty(C.safe_encode_buffer_size(n), dtype=torch.uint8, device="cuda")
    m = C.encode(d_in, d_out)                                             # lion_encode(): device pointers, synchronous (path 4)
    data = d_in.cpu().numpy()
    want, copied = oracle.encode("lion", data, return_copied=True)
    assert copied > 0
    assert m == want.size
    got = d_out[:m].cpu().numpy()
    for off in range(0, m, 1 << 28):                                      # compare in pieces: bounded temporaries
        assert (got[off:off + (1 << 28)] == want[off:off + (1 << 28)]).all(), off


@pytest.mark.parametrize("path", [0, 1])
@pytest.mark.parametrize("kind,nbytes", [("text", 5), ("text", 135), ("text", 136), ("text", 137), ("text", 300), ("text", 4096 + 3), ("text", 70001),
                                         ("text", (1 << 20) + 5), ("text", 6 * (1 << 20) + 2), ("mixed", 3 * (1 << 20) + 1), ("random", 1 << 20),
                                         ("zeros", (1 << 20) + 7), ("low", 500000), ("dickens", 200000), ("text", 33 * (1 << 20) + 66),
                                         ("smixed", 40 * (1 << 20) + 3)])
def test_cheetah_decode_parallel_paths(torch_cuda, codecs, path, kind, nbytes):
    """Cheetah decode (cheetah.rs:67-103,152-185 through codec.rs:82-126) of oracle-made streams: path 1 = the run-parallel decoder
    only (boundaries, unpack, symbolic chunk-map pass + fold, context rounds, in-order tail; no in-order fallback), path 0 = the same
    with the in-order kernel queued behind as a safety net."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    if kind == "dickens":
        data = np.fromfile(os.path.join(os.path.dirname(__file__), "golden", "dickens_200k.bin"), np.uint8)[:nbytes]
    elif kind == "text":
        data = synth.synth_text(nbytes).numpy()
    elif kind == "smixed":
        data = synth.synth_mixed(nbytes).numpy()
    else:
        data = payload(kind, nbytes, 7)
    enc = oracle.encode("cheetah", data)
    d_enc = torch.from_numpy(enc.copy()).cuda()
    d_out = torch.zeros(nbytes + 64, dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.decode_device("cheetah", d_enc, enc.size, d_out[:nbytes], d_sz, path=path)
    torch.cuda.synchronize()
    assert int(d_sz.item()) == nbytes
    assert (d_out[:nbytes].cpu().numpy() == data).all()
    assert int(d_out[nbytes:].sum().item()) == 0, "wrote past the output capacity"


def test_cheetah_round_trip_1gib_text_parallel_decoder(torch_cuda, codecs):
    """BASELINE.json configs[2] (decode half) at full size: the run-parallel decoder alone (path 1) turns the 1 GiB stream back into
    the input, on the device."""
    torch = torch_cuda
    import density_b200
    from density_b200 import synth
    n = 1 << 30
    d_in = synth.synth_text(n, device="cuda")
    d_enc = torch.zeros(codecs["cheetah"].safe_encode_buffer_size(n), dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    density_b200.encode_device("cheetah", d_in, d_enc, d_sz, path=1)
    torch.cuda.synchronize()
    m = int(d_sz.item())
    assert m > 0
    d_dec = torch.zeros(n, dtype=torch.uint8, device="cuda")
    density_b200.decode_device("cheetah", d_enc, m, d_dec, d_sz, path=1)
    torch.cuda.synchronize()
    assert int(d_sz.item()) == n
    assert torch.equal(d_dec, d_in)


def test_encode_sharded_cpp_entry_world1(torch_cuda, codecs):
    """density_b200_encode_sharded (C++: phase 1 -> fold kernel -> phase 2 -> seam verdict -> gather) with one rank: the piece and the
    gathered stream equal the oracle's; a non-quiet shard is reported, not emitted silently."""
    torch = torch_cuda
    from density_b200 import sharded, synth
    n = 5 * (1 << 20) + 1021
    data = synth.synth_text(n).numpy()
    want = oracle.encode("chameleon", data)
    enc = sharded.ShardedEncoder(torch.device("cuda"))
    d_in = torch.from_numpy(data.copy()).cuda()
    d_out = torch.zeros(codecs["chameleon"].safe_encode_buffer_size(n), dtype=torch.uint8, device="cuda")
    d_gather = torch.zeros(d_out.numel(), dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(1, dtype=torch.int64, device="cuda")
    d_fl = torch.ones(1, dtype=torch.int32, device="cuda")
    enc.encode(d_in, d_out, d_sz, d_fl, gather_root=0, d_gather=d_gather)
    torch.cuda.synchronize()
    assert int(d_fl.item()) == 0 and int(d_sz.item()) == want.size == int(enc.d_total.item())
    assert (d_out[:want.size].cpu().numpy() == want).all() and (d_gather[:want.size].cpu().numpy() == want).all()
    bad = payload("random", 1 << 20, 3)
    d_in2 = torch.from_numpy(bad.copy()).cuda()
    enc.encode(d_in2, d_out, d_sz, d_fl)
    torch.cuda.synchronize()
    assert int(d_fl.item()) != 0
    enc.close()


def _nccl_worker(rank, world, port, n_per_rank, q):
    import os, sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    import density_b200
    from density_b200 import sharded, synth
    enc = sharded.ShardedEncoder(dev)
    d_in = synth.synth_text(n_per_rank, device=dev, first_page=rank * (n_per_rank // synth.PAGE))
    cap = density_b200.Chameleon.safe_encode_buffer_size(n_per_rank)
    d_out = torch.zeros(cap, dtype=torch.uint8, device=dev)
    d_gather = torch.zeros(world * cap, dtype=torch.uint8, device=dev) if rank == 0 else None
    d_sz = torch.zeros(1, dtype=torch.int64, device=dev)
    d_fl = torch.ones(1, dtype=torch.int32, device=dev)
    enc.encode(d_in, d_out, d_sz, d_fl, gather_root=0, d_gather=d_gather)
    torch.cuda.synchronize()
    total = int(enc.d_total.item())
    q.put((rank, int(d_fl.item()), d_out[:int(d_sz.item())].cpu().numpy(), total, d_gather[:total].cpu().numpy() if rank == 0 else None))
    dist.barrier()
    enc.close()
    dist.destroy_process_group()


def test_encode_sharded_two_ranks_nccl_equals_oracle(torch_cuda, codecs):
    """Two processes, two GPUs, NCCL over NVLink: the concatenated pieces AND the stream gathered on rank 0 equal oracle.encode of the
    whole buffer (codec.rs:72-80: one stream). Skipped on a single-GPU box (the driver's 2 / 4 / 8-GPU bench runs the same check)."""
    torch = torch_cuda
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from density_b200 import synth
    world, n_per = 2, 48 * (1 << 20)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, world, 29713, n_per, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(world):
        r, fl, piece, total, gathered = q.get(timeout=600)
        got[r] = (fl, piece, total, gathered)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    whole = synth.synth_text(world * n_per).numpy()
    want = oracle.encode("chameleon", whole)
    assert all(got[r][0] == 0 for r in range(world))
    cat = np.concatenate([got[r][1] for r in range(world)])
    assert cat.size == want.size and (cat == want).all()
    assert got[0][2] == want.size and (got[0][3] == want).all()


@pytest.mark.parametrize("alg", ALGS)
def test_codec_instance_streaming_continuation(torch_cuda, codecs, alg):
    """density_b200_codec_* (a reused Codec instance, codec.rs:16,72,82) against an oracle instance that is reused the same way: three
    pieces encoded one after the other (text, a piece with copy-mode blocks, text again), decoded by a second instance, then
    clear_state() and a fresh start. Chameleon encode takes the run-parallel kernels with the dictionary carried in."""
    from density_b200.codec import CodecInstance
    from density_b200 import synth
    big = alg == "chameleon"
    pieces = [synth.synth_text((3 << 20) + 5 if big else 150001).numpy(),
              synth.synth_mixed((2 << 20) + 256 * 3 if big else 120000).numpy(),
              synth.synth_text((1 << 20) + 77 if big else 70001, first_page=9).numpy()]
    want_inst = oracle.Codec(alg)
    enc, dec = CodecInstance(alg), CodecInstance(alg)
    streams = []
    for p in pieces:
        want = want_inst.encode(p)
        out = np.zeros(codecs[alg].safe_encode_buffer_size(p.size), dtype=np.uint8)
        n = enc.encode(p, out)
        assert n == want.size and (out[:n] == want).all(), (alg, p.size)
        streams.append(out[:n].copy())
    for p, s in zip(pieces, streams):
        back = np.zeros(p.size, dtype=np.uint8)
        assert dec.decode(s, back) == p.size and (back == p).all()
    enc.clear_state()
    out = np.zeros(codecs[alg].safe_encode_buffer_size(pieces[2].size), dtype=np.uint8)
    n = enc.encode(pieces[2], out)
    want = oracle.encode(alg, pieces[2])
    assert n == want.size and (out[:n] == want).all()
    enc.close(); dec.close()
