#!/usr/bin/env python
"""bench.py — headline benchmark of the density_b200 hot path (see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU (oracle port)

A "step" is one Chameleon encode of one synthetic-text buffer (BASELINE.json configs[1]: 1 GiB per GPU, resident in HBM
when the timed region starts). Metric: input GB/s (uncompressed bytes / time, GB = 1e9 B — the reference's own convention,
/root/reference/benches/density.rs:29,48). N>1: one process per GPU (torchrun), every rank owns one 1 GiB shard of ONE
bit-exact stream; the only collective is the all_gather of the 256 KiB dictionary tables (weak scaling).
Rank 0 prints ONE JSON line.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GiB = 1 << 30
METRIC = "chameleon_encode_input_GBps"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--bytes", type=int, default=GiB, help="bytes per GPU (default 1 GiB: BASELINE.json configs[1])")
    ap.add_argument("--cpu-sample-bytes", type=int, default=256 << 20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the oracle digest check of the produced stream (outside the timed region)")
    ap.add_argument("--no-config5", action="store_true", help="N > 1: skip the 8 GiB-per-GPU encode-only / gather-inclusive extra")
    ap.add_argument("--config5-bytes", type=int, default=8 * GiB)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's output (stream size and a seeded sample of the stream) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def time_oracle(sample, repeats):
    """Reference algorithm (oracle port, oracle/density_oracle.c) on ONE host core: the reference is single-threaded
    (README.md:42) and one stream cannot be split without changing its bytes."""
    import numpy as np
    import oracle
    L = oracle.lib()
    cap = oracle.safe_encode_buffer_size("chameleon", sample.size)
    out = np.zeros(cap, dtype=np.uint8)      # pre-faulted: page faults are not part of the codec
    L.oracle_encode(0, sample.ctypes.data, min(sample.size, 8 << 20), out.ctypes.data, cap)  # untimed warm-up
    times = []
    for _ in range(repeats):
        t = time.perf_counter()
        n = L.oracle_encode(0, sample.ctypes.data, sample.size, out.ctypes.data, cap)
        times.append(time.perf_counter() - t)
        assert n > 0
    return times, n


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    from density_b200 import synth
    nb = min(args.bytes, args.cpu_sample_bytes)
    sample = synth.synth_text(nb).numpy()
    time_oracle(sample[: min(nb, 16 << 20)], max(1, min(args.warmup, 3)))
    times, n = time_oracle(sample, args.steps)
    tot = sum(times)
    val = nb * len(times) / tot / 1e9
    cores = 1
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "Chameleon encode, synthetic English text (BASELINE.json configs[1])", "bytes_per_step": nb,
                   "note": "reference algorithm restated in C (oracle/density_oracle.c; no Rust toolchain on the box), "
                           "1 thread: the reference is single-threaded and one stream cannot be split bit-exactly"},
        "cpu_baseline": {"value": val, "unit": "GB/s", "cores": cores, "kind": "port",
                         "sample": f"{nb >> 20} MiB prefix of the 1 GiB synthetic-text workload per step"},
        "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host_cpus": os.cpu_count(), "ratio": sample.size / n,
    }
    print(json.dumps(line))


def _sha(t):
    import hashlib
    return hashlib.sha256(t.cpu().numpy().tobytes()).hexdigest()


def verify_against_oracle(dev, world, rank, n, d_out, out_bytes, dist, torch, synth):
    """Outside the timed region: every rank hashes its piece; rank 0 regenerates the WHOLE input (world x n bytes of the same
    counter-based text), runs the oracle over it in one call and compares the digests of the oracle's stream, cut at the ranks' sizes,
    with the ranks' digests (codec.rs:72-80: one stream). Returns a dict for the JSON line; raises on a mismatch."""
    import hashlib
    import numpy as np
    import oracle
    mine = hashlib.sha256(d_out[:out_bytes].cpu().numpy().tobytes()).hexdigest()
    if world > 1:
        objs = [None] * world
        dist.all_gather_object(objs, (int(out_bytes), mine))
    else:
        objs = [(int(out_bytes), mine)]
    res = None
    if rank == 0:
        whole = np.empty(world * n, dtype=np.uint8)
        for r in range(world):
            whole[r * n:(r + 1) * n] = synth.synth_text(n, device=dev, first_page=r * (n // synth.PAGE)).cpu().numpy()
        t0 = time.perf_counter()
        want = oracle.encode("chameleon", whole)
        dt = time.perf_counter() - t0
        off = 0
        ok = want.size == sum(sz for sz, _ in objs)
        for r, (sz, dig) in enumerate(objs):
            piece = want[off:off + sz]
            ok = ok and hashlib.sha256(piece.tobytes()).hexdigest() == dig
            off += sz
        res = {"checked": True, "ok": bool(ok), "bytes": int(world * n), "stream_bytes": int(want.size), "oracle_s": round(dt, 2),
               "how": "sha256 of every rank's piece == the oracle's single-call stream cut at the ranks' sizes"}
        if not ok:
            raise SystemExit("bench.py: the sharded stream differs from the oracle's: " + json.dumps(res))
    return res


DUMP_WINDOWS, DUMP_WINDOW_BYTES = 1024, 8192     # 8 MiB of stream over all ranks, 32 MiB as float32


def dump_outputs(dirname, suffix, d_out, out_bytes, windows, d_flags=None):
    """What a caller of the timed path receives: the encoded size, the stream and (sharded) the flags, as float arrays. A stream
    longer than `windows` x DUMP_WINDOW_BYTES is sampled in windows at offsets drawn from a fixed seed, so that two builds run
    with the same arguments are compared on the same bytes."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    if out_bytes <= windows * DUMP_WINDOW_BYTES:
        offs = np.zeros(1, dtype=np.int64)
        sample = d_out[:out_bytes][None]
    else:
        offs = np.sort(np.random.default_rng(0).integers(0, out_bytes - DUMP_WINDOW_BYTES + 1, size=windows))
        idx = torch.from_numpy(offs).to(d_out.device)[:, None] + torch.arange(DUMP_WINDOW_BYTES, device=d_out.device)
        sample = d_out[idx]
    arrays = {"stream_size": np.array([out_bytes], dtype=np.float64), "stream_sample": sample.float().cpu().numpy(),
              "stream_sample_offsets": offs.astype(np.float64)}
    if d_flags is not None:
        arrays["flags"] = d_flags.double().cpu().numpy()
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + suffix + ".npy"), a)


def cpu_rate(alg, op, sample, reps=3):
    """oracle port on one host core: input GB/s (uncompressed bytes / time, benches/density.rs:29,48)"""
    import numpy as np
    import oracle
    L = oracle.lib()
    cap = oracle.safe_encode_buffer_size(alg, sample.size)
    enc = np.zeros(cap, dtype=np.uint8)
    m = L.oracle_encode(oracle.ALGS[alg], sample.ctypes.data, sample.size, enc.ctypes.data, cap)
    dec = np.zeros(sample.size + 8, dtype=np.uint8)
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        if op == "encode":
            L.oracle_encode(oracle.ALGS[alg], sample.ctypes.data, sample.size, enc.ctypes.data, cap)
        else:
            L.oracle_decode(oracle.ALGS[alg], enc.ctypes.data, m, dec.ctypes.data, sample.size)
        ts.append(time.perf_counter() - t)
    return sample.size / min(ts) / 1e9


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import density_b200
    from density_b200 import synth, sharded

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the density_b200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # keep rank 0's stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    L = density_b200.load()
    C = density_b200.Chameleon
    n = args.bytes
    assert n % 256 == 0
    peak_gbs, peak_src = measured_peaks()

    # ---- workload: rank r owns pages [r*n/64Ki, ...) of the infinite synthetic corpus: one contiguous stream ----------
    d_in = synth.synth_text(n, device=dev, first_page=rank * (n // synth.PAGE))
    cap = C.safe_encode_buffer_size(n)
    d_out = torch.empty(cap, dtype=torch.uint8, device=dev)
    d_size = torch.zeros(1, dtype=torch.int64, device=dev)
    d_flags = torch.zeros(1, dtype=torch.int32, device=dev)
    enc = sharded.ShardedEncoder(dev) if world > 1 else None     # C++: density_b200_encode_sharded (NCCL inside the library)

    def step():
        if world > 1:
            enc.encode(d_in, d_out, d_size, d_flags)
        else:
            density_b200.encode_device("chameleon", d_in, d_out, d_size)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    L.density_b200_profile_enable(1 if world == 1 else 0)
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    out_bytes = int(d_size.item())
    assert out_bytes > 0
    if world == 1:
        assert L.density_b200_last_encode_was_fast() == 1, "synthetic text must take the segment-parallel path"
    else:
        assert int(d_flags.item()) == 0

    # ---- timed region: device-resident, CUDA events on the launching stream, inputs (1 GiB) >> L2 (126 MB) ---------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = L.density_b200_kernel_launches()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    stage_ms = np.zeros(5)
    barrier()
    L.density_b200_profile_enable(1 if world == 1 else 0)   # reset the per-stage event ring: it now covers exactly the timed steps
    ev[0].record()
    for i in range(args.steps):
        step()
        ev[i + 1].record()
    barrier()
    prof = (ctypes.c_float * 3)()
    if world == 1 and L.density_b200_profile_get(prof) != 0:
        raise SystemExit("profile_get failed: " + density_b200._lib.last_error())
    if world > 1:
        stage_ms = np.array(enc.profile())                   # last timed step (every step is the same work)
    total_ms = ev[0].elapsed_time(ev[args.steps])
    launches = L.density_b200_kernel_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([total_ms] + list(stage_ms), dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t[0].item())
    stage_ms = [float(x) for x in t[1:].tolist()]
    ms_per_step = total_ms / args.steps
    value = world * n / (ms_per_step * 1e-3) / 1e9
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, f"_rank{rank}" if world > 1 else "", d_out, int(d_size.item()), DUMP_WINDOWS // world,
                     d_flags if world > 1 else None)

    # ---- parity, outside the timed region: the stream(s) just produced against ONE oracle call over the whole input --------------
    parity = None
    if not args.no_verify:
        parity = verify_against_oracle(dev, world, rank, n, d_out, out_bytes, dist, torch, synth)

    # ---- e2e: the reference-facing symbol chameleon_encode() with HOST (pinned) buffers, copies inside the timing ---
    e2e = None
    e2e_extra = {}
    if not args.no_e2e:
        h_in = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        h_in.copy_(d_in)
        h_out = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
        a_in, a_out = h_in.numpy(), h_out.numpy()
        h_size = torch.zeros(1, dtype=torch.int64, pin_memory=True)

        def e2e_step():
            if world == 1:
                return C.encode(a_in, a_out)          # reference-shaped C ABI symbol, host pointers
            # N > 1: the public sharded API, same host buffers; H2D / D2H copies are part of the step
            d_in.copy_(h_in, non_blocking=True)
            enc.encode(d_in, d_out, d_size, d_flags)
            h_size.copy_(d_size, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            mm = int(h_size.item())
            h_out[:mm].copy_(d_out[:mm], non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return mm

        for _ in range(3):
            m = e2e_step()
        assert m == out_bytes
        k = max(3, min(args.steps, 10))
        barrier()
        t0 = time.perf_counter()
        for _ in range(k):
            m = e2e_step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * n * k / float(tt.item()) / 1e9, "unit": "GB/s", "h2d_bytes_per_step": n, "d2h_bytes_per_step": int(m) + 8,
               "steps": k, "api": ("chameleon_encode(host ptr, n, host ptr, cap): C ABI, pinned host buffers, synchronous" if world == 1 else
                                   "density_b200_encode_sharded with pinned host buffers: H2D + phase 1 + ncclAllGather + phase 2 + D2H per step (no overlap)")}
        if world == 1:
            # what a caller with ordinary (pageable) memory sees — a Rust Vec<u8> is pageable — and the decode direction
            p_in = np.empty(n, dtype=np.uint8); p_in[:] = a_in
            p_out = np.zeros(cap, dtype=np.uint8)
            C.encode(p_in, p_out)
            t0 = time.perf_counter()
            for _ in range(3):
                mm = C.encode(p_in, p_out)
            e2e_extra["chameleon_encode_pageable_GBps"] = 3 * n / (time.perf_counter() - t0) / 1e9
            assert mm == out_bytes
            h_dec = torch.empty(n, dtype=torch.uint8, pin_memory=True)
            a_dec = h_dec.numpy()
            C.decode(a_out[:out_bytes], a_dec)
            t0 = time.perf_counter()
            for _ in range(3):
                dn = C.decode(a_out[:out_bytes], a_dec)
            e2e_extra["chameleon_decode_pinned_GBps"] = 3 * n / (time.perf_counter() - t0) / 1e9
            assert dn == n and bool((h_dec == h_in).all())
            e2e_extra["note"] = "input GB/s through the nine reference symbols with HOST buffers; H2D + D2H inside the timing"
            del p_in, p_out, h_dec

    # ---- extra (not the headline metric): the other BASELINE.json configurations, device-resident, N=1 only ----------------------
    extra = None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, reps):
        fn(); torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    if world == 1:
        d_dec = torch.empty(n, dtype=torch.uint8, device=dev)
        d_dsz = torch.zeros(1, dtype=torch.int64, device=dev)
        density_b200.decode_device("chameleon", d_out, out_bytes, d_dec, d_dsz)
        torch.cuda.synchronize()
        assert int(d_dsz.item()) == n and torch.equal(d_dec, d_in), "decode(encode(x)) != x"
        dms = timed(lambda: density_b200.decode_device("chameleon", d_out, out_bytes, d_dec, d_dsz), max(3, min(args.steps, 10)))
        extra = {"chameleon_decode_GBps": n / (dms * 1e-3) / 1e9, "decode_ms": dms, "round_trip_verified": True,
                 "chameleon_decode_roofline_frac": (n + out_bytes) / (dms * 1e-3) / 1e9 / peak_gbs,
                 "note": "uncompressed bytes / time, same convention as the reference's decompress bench (benches/density.rs:48); "
                         "roofline fractions = (stream + original bytes) / time / measured HBM peak"}
        # config 3 (Cheetah encode + decode, 1 GiB text) and Lion encode on the same buffer; bit-exactness at these sizes is the tests' job
        for alg in ("cheetah", "lion"):
            C2 = density_b200.CODECS[alg]
            d_o2 = torch.empty(C2.safe_encode_buffer_size(n), dtype=torch.uint8, device=dev)
            d_s2 = torch.zeros(1, dtype=torch.int64, device=dev)
            ams = timed(lambda: density_b200.encode_device(alg, d_in, d_o2, d_s2, path=1), 3)
            m2 = int(d_s2.item())
            assert m2 > 0, f"{alg}: copy map did not settle on the bench input"
            extra[f"{alg}_encode_GBps"] = n / (ams * 1e-3) / 1e9
            extra[f"{alg}_encode_ms"] = ams
            extra[f"{alg}_ratio"] = n / m2
            extra[f"{alg}_encode_roofline_frac"] = (n + m2) / (ams * 1e-3) / 1e9 / peak_gbs
            if alg == "cheetah":
                d_dsz.zero_()
                cms = timed(lambda: density_b200.decode_device("cheetah", d_o2, m2, d_dec, d_dsz, path=1), 3)
                ok = int(d_dsz.item()) == n and torch.equal(d_dec, d_in)
                extra["cheetah_decode_GBps"] = n / (cms * 1e-3) / 1e9
                extra["cheetah_decode_ms"] = cms
                extra["cheetah_decode_round_trip_verified"] = bool(ok)
                extra["cheetah_decode_roofline_frac"] = (n + m2) / (cms * 1e-3) / 1e9 / peak_gbs
                assert ok, "cheetah: parallel decode(encode(x)) != x"
            del d_o2
        del d_dec
        # Chameleon encode of data on which the protection automaton fires (copy-mode blocks): 256 MiB of noise and of mixed text / binary
        for kind, gen in (("noise", lambda k: synth.random_bytes(k, 5, device=dev)), ("mixed", lambda k: synth.synth_mixed(k, device=dev))):
            nk = 256 << 20
            d_k = gen(nk)
            d_ok = torch.empty(density_b200.Chameleon.safe_encode_buffer_size(nk), dtype=torch.uint8, device=dev)
            kms = timed(lambda: density_b200.encode_device("chameleon", d_k, d_ok, d_dsz), 3)
            extra[f"chameleon_encode_{kind}_256MiB_GBps"] = nk / (kms * 1e-3) / 1e9
            extra[f"chameleon_encode_{kind}_256MiB_ratio"] = nk / max(int(d_dsz.item()), 1)
            del d_k, d_ok
        # config 1: Chameleon round trip on Silesia/dickens through the reference symbols (latency-bound on a GPU; reported, not optimised)
        dk = None
        # the file: $FILE as in the reference's benches (utils.rs:6-17), else the first 200,003 B of dickens kept in the tree
        cands = [(os.path.join(ROOT, "tests", "golden", "dickens_200k.bin"), "first 200,003 B of dickens (tests/golden)")]
        if os.environ.get("FILE"):
            cands.insert(0, (os.environ["FILE"], "FILE=" + os.environ["FILE"]))
        for cand, label in cands:
            if os.path.exists(cand):
                dk, dk_label = np.fromfile(cand, dtype=np.uint8), label
                break
        if dk is not None:
            dko = np.zeros(C.safe_encode_buffer_size(dk.size), dtype=np.uint8)
            dkd = np.zeros(dk.size, dtype=np.uint8)
            mdk = C.encode(dk, dko); C.decode(dko[:mdk], dkd)
            assert bool((dkd == dk).all())
            reps = 10
            t0 = time.perf_counter()
            for _ in range(reps):
                C.encode(dk, dko)
            te = (time.perf_counter() - t0) / reps
            t0 = time.perf_counter()
            for _ in range(reps):
                C.decode(dko[:mdk], dkd)
            td = (time.perf_counter() - t0) / reps
            extra["config1_dickens"] = {"file": dk_label, "ratio": dk.size / mdk, "gpu_encode_GBps": dk.size / te / 1e9, "gpu_decode_GBps": dk.size / td / 1e9,
                                        "cpu_encode_GBps": cpu_rate("chameleon", "encode", dk, 5), "cpu_decode_GBps": cpu_rate("chameleon", "decode", dk, 5),
                                        "note": "host buffers through chameleon_encode / chameleon_decode (copies included), next to the oracle port on one core; "
                                                "the reference publishes 2.156 / 2.952 GB/s for this file (benchmark.log:18,20)"}
        extra.update(e2e_extra)

    # ---- config 5 (N > 1): 8 GiB per GPU, encode-only and gather-inclusive ------------------------------------------------------------
    cfg5 = None
    if world > 1 and not args.no_config5:
        n5 = args.config5_bytes
        free = torch.cuda.mem_get_info()[0]
        need = 2.2 * n5 + (0.6 * n5 * world if rank == 0 else 0) + (2 << 30)
        fits = torch.tensor([1 if free > need else 0], device=dev)
        dist.all_reduce(fits, op=dist.ReduceOp.MIN)
        if int(fits.item()) == 1:
            del d_in, d_out
            torch.cuda.empty_cache()
            d_in5 = torch.empty(n5, dtype=torch.uint8, device=dev)
            for off in range(0, n5, 1 << 30):
                kk = min(1 << 30, n5 - off)
                d_in5[off:off + kk] = synth.synth_text(kk, device=dev, first_page=(rank * n5 + off) // synth.PAGE)
            d_out5 = torch.empty(C.safe_encode_buffer_size(n5), dtype=torch.uint8, device=dev)
            d_gather = torch.empty(int(0.6 * n5 * world), dtype=torch.uint8, device=dev) if rank == 0 else None

            def run5(gather):
                enc.encode(d_in5, d_out5, d_size, d_flags, gather_root=0 if gather else -1, d_gather=d_gather)

            res5 = {}
            for name, g in (("encode_only", False), ("with_gather", True)):
                for _ in range(2):
                    run5(g)
                barrier()
                e0.record()
                for _ in range(3):
                    run5(g)
                e1.record()
                barrier()
                tms = torch.tensor([e0.elapsed_time(e1) / 3], dtype=torch.float64, device=dev)
                dist.all_reduce(tms, op=dist.ReduceOp.MAX)
                res5[name + "_ms"] = float(tms.item())
                res5[name + "_GBps"] = world * n5 / (float(tms.item()) * 1e-3) / 1e9
            assert int(d_flags.item()) == 0
            total5 = int(enc.d_total.item())
            res5.update({"bytes_per_gpu": n5, "total_bytes": world * n5, "stream_bytes": total5,
                         "gather": "pieces to rank 0 at prefix-sum offsets: grouped ncclSend / ncclRecv (root-inbound NVLink bound)",
                         "gather_GBps_of_stream": (total5 * (world - 1) / world) / max(1e-9, (res5["with_gather_ms"] - res5["encode_only_ms"]) * 1e-3) / 1e9})
            if rank == 0:
                # the gathered stream must be one stream: its first 64 MiB of input decode back from its head (size-independent check)
                npre = 64 << 20
                d_dec = torch.empty(npre + 4096, dtype=torch.uint8, device=dev)
                import oracle
                want = oracle.encode("chameleon", d_in5[:npre].cpu().numpy())
                res5["gathered_head_matches_oracle"] = bool((d_gather[:want.size - 300].cpu().numpy() == want[:want.size - 300]).all())
                assert res5["gathered_head_matches_oracle"]
                del d_dec
            cfg5 = res5

    # ---- CPU baseline (rank 0) -------------------------------------------------------------------------------------------------------
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        nb = min(n, args.cpu_sample_bytes)
        sample = synth.synth_text(nb, device=dev).cpu().numpy()
        time_oracle(sample[: 16 << 20], 1)
        reps = 8 if world == 1 else 4
        times, _ = time_oracle(sample, reps)
        cpu = {"value": nb * reps / sum(times) / 1e9, "unit": "GB/s", "cores": 1, "kind": "port",
               "sample": f"{nb >> 20} MiB prefix of the step's buffer x {reps} (oracle/density_oracle.c, 1 thread; host has {os.cpu_count()} CPUs)"}
        if world == 1 and extra is not None:
            small = sample[: 64 << 20]
            extra["cpu_baselines_GBps"] = {f"{a}_{op}": cpu_rate(a, op, small, 2) for a in ("chameleon", "cheetah", "lion") for op in ("encode", "decode")}
            extra["cpu_baselines_GBps"]["sample"] = "64 MiB of the bench text, oracle port, 1 core, best of 2"

    if rank != 0:
        if world > 1:
            enc.close()
            dist.destroy_process_group()
        return
    line = {
        "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
        "data": "synthetic",
        "config": {"workload": "Chameleon encode, 1 GiB synthetic English text per GPU (BASELINE.json configs[1])",
                   "bytes_per_gpu": n, "out_bytes_rank0": out_bytes, "ratio": n / out_bytes,
                   "l2_policy": "input 1 GiB + output 0.57 GiB per step >> 126 MB L2 (no flush needed)",
                   "parallelism": (f"{world} shards of one bit-exact stream (density_b200_encode_sharded, C++): ncclAllGather of 256 KiB tables + "
                                   "32-byte seam words; pieces stay on their GPUs in `value` (gather-inclusive: config5)") if world > 1 else "single GPU"},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if e2e:
        line["e2e"] = e2e
    if parity:
        line["parity"] = parity
    sig = n / 32
    step_alg = (n + out_bytes) / (ms_per_step * 1e-3) / 1e9
    if world == 1:
        fp, mid, em = [float(x) for x in prof]
        exch = 0.0
    else:
        fp, exch, mid, em = stage_ms[0], stage_ms[1], stage_ms[2], stage_ms[3]
    kernels = {
        "cham_flag_pass": {"ms": fp, "alg_bytes": n + sig, "gbs": (n + sig) / (fp * 1e-3) / 1e9 if fp > 0 else None},
        "cham_emit": {"ms": em, "alg_bytes": n + sig + out_bytes, "gbs": (n + sig + out_bytes) / (em * 1e-3) / 1e9 if em > 0 else None},
        "carry_resolve_sizes_scan": {"ms": mid},
    }
    if world > 1:
        kernels["table_allgather_and_fold"] = {"ms": exch}
        kernels["seam_words_allgather"] = {"ms": stage_ms[4]}
    dom = "cham_flag_pass" if fp >= em else "cham_emit"
    ach = kernels[dom]["gbs"]
    traffic = None   # dram__bytes_read.sum + dram__bytes_write.sum of that kernel from the committed ncu --set full capture
    try:
        if n == GiB:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))["dram_bytes_per_launch"][dom]
    except Exception:
        traffic = None
    line["roofline"] = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak_gbs, "unit": "GB/s",
                        "frac": (ach / peak_gbs) if ach else None, "traffic": traffic, "peak_source": peak_src,
                        "per": "one GPU (max over ranks of the stage times)" if world > 1 else "one GPU",
                        "step_algorithmic": {"bytes": n + out_bytes, "achieved": step_alg / world, "frac": step_alg / world / peak_gbs},
                        "input_rate_frac": value / world / peak_gbs, "kernels": kernels}
    if extra:
        line["extra"] = extra
    if cfg5:
        line.setdefault("extra", {})["config5"] = cfg5
    if cpu:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))
    if world > 1:
        enc.close()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
