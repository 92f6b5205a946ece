#!/usr/bin/env python
"""Benchmark of the hot path: ct x ct fhe_multiply + relinearisation (BASELINE.json `metric`).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine (one process per GPU)
  python bench.py --impl reference --gpus N --steps K ...   # the CPU restatement of the SEAL path (oracle/)

A "step" is one pass of the hot path over one batch of 4,096 synthetic ciphertext pairs per GPU
(BASELINE.json configs[2]).  `value` = whole-job ops/s with inputs resident in HBM; `e2e` = the same metric
through the C-ABI host-buffer entry point (fhe_b200_mul_relin_host: pinned host limb arrays in, H2D + kernels
+ D2H inside the timed region).  One JSON line on stdout from rank 0.  `--dump-outputs DIR` also writes a fixed sample of
the last timed step's results as .npy files, to compare two builds output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N = 4096
Q = (0xFFFFEE001, 0xFFFFC4001)
CT_BYTES = 2 * 2 * N * 8  # 131,072
ALGO_BYTES_PER_OP = 3 * CT_BYTES  # SURVEY 8(d): read a, read b, write result = 393,216 B
# SURVEY 8(d): SEAL's form runs 47 limb-NTTs x 24,576 butterflies per op.  The library computes the same bits three ways
# (FHE_B200_BEHZ, DESIGN.md section 4): "dual" (default) carries the BEHZ tensor product on six primes below 2^30, two per
# 64-bit word (21 dual transforms + 12 key-switch transforms); "bsk" on SEAL's three 61-bit primes with the q-limbs recovered
# from them (33 transforms); "seal" transforms the q-limbs too (47).
BEHZ = "seal" if os.environ.get("FHE_B200_QLIMB_NTT") == "1" else os.environ.get("FHE_B200_BEHZ", "dual")
if BEHZ not in ("dual", "bsk", "seal"):
    BEHZ = "dual"
QLIMB_NTT = BEHZ == "seal"
NTTS_PER_OP = 47 if QLIMB_NTT else 33
BUTTERFLIES_PER_OP = NTTS_PER_OP * 24576
# Integer-pipe roofline.  The binding resource is the SM's 32-bit multiplier (the "heavy" half of the FMA pipe): IMAD.WIDE /
# IMAD.HI issue at 32 results per clock per SM (quarter rate), IMAD at 64 (half rate = 0.5 IMAD.WIDE-equivalents).
# ALGORITHMIC multiplier work of one ct x ct multiply + relinearise, in IMAD.WIDE-equivalents -- the cheapest exact
# formulation we know on a 32-bit multiplier, independent of how a kernel happens to be scheduled (DESIGN.md section 4):
#   one Shoup butterfly X +- w Y by a precomputed (w, floor(w 2^64 / q)):
#     36/37-bit primes, forward : quotient estimate 2 wide + 1 low, low product 1 wide + 2 low, -H q 1 wide + 2 low = 4 w + 5 l = 6.5
#     36/37-bit primes, inverse : operand range 2^51 needs one more partial product of the quotient            = 5 w + 4 l = 7.0
#     61-bit primes             : exact quotient 4 partial products (the lowest feeds one carry), low product 1 w + 2 l,
#                                 -H q as H c - (H << 61): 1 w + 1 l                                            = 6 w + 3 l = 7.5
#   NTTs per op, SEAL's form (FHE_B200_QLIMB_NTT=1): 14 forward + 12 inverse on 36/37-bit primes, 12 forward + 9 inverse on
#   61-bit primes (SURVEY 8d: 26 + 21).  Default: the 8 forward + 6 inverse q-limb transforms of the tensor product are not run
#   (6 + 6 on 36/37-bit primes, 12 + 9 on 61-bit primes); k_floor_sk recovers them exactly (3 Shoup products by constants + two
#   3-term sums of Shoup products) and lifts the floor result from (b0, b1) by exact rounding instead of Shenoy-Kumaresan's
#   m_sk correction: 98.5 IMAD.WIDE-equivalents per coefficient (5 x 6.5 Shoup products, 10 x 5 sum terms, 4 x 1.5 small
#   terms, 4 x 1.5 reductions, 4 for the punctured sum and its folds) against 113 for SEAL's step-by-step form.
#   pointwise (base conversions in the integer domain, tensor, key-switch MAC, division by P), per kernel below.
# Per kernel (what bench.py's live CUDA-event timing is divided into):
if BEHZ == "seal":
    KERNEL_WIDE_EQ = {
        "k_ext_conv": 42.5 * 16384,                                  # fastbconv_m_tilde + sm_mrq per coefficient of the 4 input polys
        "k_ext_ntt": 24576 * (8 * 6.5 + 12 * 7.5),                   # 20 forward NTTs: 8 on q limbs, 12 on the Bsk limbs
        "k_tensor_intt": 24576 * (6 * 7.0 + 9 * 7.5) + 0.51e6,       # 15 inverse NTTs + the dyadic tensor
        "k_floor_sk": 113.0 * 12288,                                 # fast_floor + fastbconv_sk per coefficient of the 3 output polys
    }
elif BEHZ == "bsk":
    KERNEL_WIDE_EQ = {
        "k_ext_conv": 42.5 * 16384,                                  # fastbconv_m_tilde + sm_mrq per coefficient of the 4 input polys
        "k_ext_ntt": 24576 * 12 * 7.5,                               # 12 forward NTTs on the Bsk limbs
        "k_tensor_intt": 24576 * 9 * 7.5 + 0.36e6,                   # 9 inverse NTTs + the dyadic tensor on the Bsk limbs
        "k_floor_sk": 98.5 * 12288,                                  # q-limb recovery + fast_floor + exact lift from (b0, b1) per coefficient
    }
else:
    # dual base: one butterfly = two 32-bit Shoup products (IMAD.HI + 2 IMAD each) = 4 IMAD.WIDE-equivalents for both lanes
    KERNEL_WIDE_EQ = {
        "k_ext_conv": (36.5 + 6 * 3.5) * 16384,                      # shared part of the extension + 6 residues (2 wide + Barrett each)
        "k_ext_ntt": 24576 * 12 * 4.0,                               # 12 forward dual transforms
        "k_tensor_intt": 24576 * 9 * 4.0 + 9 * 2048 * 4.0 + 17.0 * 12288,  # 9 inverse dual transforms (scaled last stage) + dyadic tensor
        # 6 Shoup products on 32 bits (2.0 each), 12 + 8 terms of exact two-accumulator sums (2 wide each, WideSum), 4 reductions of
        # such sums (4.0), the punctured sum (6), y0 mod 4 primes and the 4-prime lift (4.5 each): 92 per coefficient; it was 115
        # while the sums were sums of Shoup products (3 wide + 1 low per term)
        "k_floor_sk": 92.0 * 12288,
    }
# key switch: "dual" (default for chunks >= 96 ops) carries switch_key_inplace's sums on the dual base too -- 6 + 6 dual transforms
# and one CRT recovery per output coefficient; "seal" runs the 6 + 6 transforms on SEAL's key primes q0, q1, P
KS = "seal" if os.environ.get("FHE_B200_KS") == "seal" else "dual"
KERNEL_WIDE_EQ.update({
    "k_digit_ntt": 24576 * 6 * 6.5,                              # 6 key-switch digit NTTs
    "k_ks_finish": 24576 * 6 * 7.0 + 0.28e6 + 0.13e6,            # key MAC + 6 inverse NTTs + rounded division by P
    "k_digit_ntt_ksd": 24576 * 6 * 4.0 + 2 * 4096 * 6 * 1.5,     # 6 forward dual transforms + the digits reduced mod the six primes
    "k_ks_intt_ksd": 24576 * 6 * 4.0 + 6 * 2048 * 4.0 + 3.5 * 2 * 4096 * 6,  # 6 inverse dual transforms (scaled last stage) + key MAC
    # 6 Shoup products on 32 bits (2.0), U mod P (6 sum terms x 2 + 4), then per q-limb 7 sum terms (the P^-1-scaled CRT terms and
    # the low part of the P-limb correction) + 2 small terms + one reduction: 68 per coefficient of the two output polynomials
    "k_ks_finish_ksd": 68.0 * 8192,
})
# the fused tails (default; FHE_B200_FUSE_TAIL=0 splits them): the same arithmetic without the HBM round trip of the tensor product / of U_k
FUSE_TAIL = int(os.environ.get("FHE_B200_FUSE_TAIL", "3"))
KERNEL_WIDE_EQ["k_tensor_floor_d"] = KERNEL_WIDE_EQ["k_tensor_intt"] + KERNEL_WIDE_EQ["k_floor_sk"]
KERNEL_WIDE_EQ["k_ks_tail_ksd"] = KERNEL_WIDE_EQ["k_ks_intt_ksd"] + KERNEL_WIDE_EQ["k_ks_finish_ksd"]
KERNEL_WIDE_EQ["k_ks_intt"] = 24576 * 6 * 7.0 + 0.28e6           # the unfused tail (small chunks): MAC + inverse NTTs
KERNEL_WIDE_EQ["k_relin_finish"] = 0.13e6                        #   ... and the division by P
KS_KERNELS = ("k_digit_ntt_ksd", "k_ks_intt_ksd", "k_ks_finish_ksd") if KS == "dual" else ("k_digit_ntt", "k_ks_finish")
WIDE_EQ_PER_OP = sum(KERNEL_WIDE_EQ[k] for k in ("k_ext_conv", "k_ext_ntt", "k_tensor_intt", "k_floor_sk") + KS_KERNELS)  # fusing changes no count
SM_COUNT = 148
WIDE_PER_CLK_PER_SM = 32  # IMAD.WIDE results per clock per SM (scripts/pipe_probe.cu: 0.25 warp-instructions / clk / SMSP)
METRIC = "ct_ct_fhe_multiply_relin_ops_per_sec"
WORKLOAD = "batch of 4096 ct*ct fhe_multiply+relinearize per GPU, testnet BFV params (N=4096, q=72b, t=4096)"
DUMP_ROWS = 256  # ciphertexts kept by --dump-outputs: 256 x 128 KiB of float64 = 32 MiB


def dump_outputs(path: str, n: int, take) -> None:
    """--dump-outputs: a fixed sample of the results of the last timed step, so that two builds can be compared output for
    output.  ct_out.npy: float64 [rows, 2, 2, 4096], the result ciphertexts (residues < 2^37, exact in float64);
    ct_out_rows.npy: the batch index of each row (DUMP_ROWS indices drawn with seed 0, ascending; the whole batch if smaller).
    `take(rows)` returns those rows of the result as uint64."""
    import numpy as np

    rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_ROWS), replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "ct_out.npy"), take(rows).astype(np.float64))
    np.save(os.path.join(path, "ct_out_rows.npy"), rows.astype(np.float64))


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int) -> None:
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self) -> None:
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def stop(self) -> dict:
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=1.0)
        s = sorted(self.samples)
        return {
            "sm_mhz": s[len(s) // 2] if s else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(s),
        }


def bind_to_gpu_numa_node(index: int) -> None:
    """Pin this rank to the CPUs local to its GPU (NVML affinity) so pinned staging memory is first-touched on the
    GPU's NUMA node; matters for the host-buffer (e2e) path when 8 ranks share the box."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        local = {64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
        allowed = os.sched_getaffinity(0) & local
        if allowed:
            os.sched_setaffinity(0, allowed)
    except Exception:
        pass


def synth_ciphertexts(torch, n: int, seed: int, device) -> "torch.Tensor":
    """[n,2,2,4096] int64: uniform residues mod (q0, q1) -- synthetic data-level ciphertexts."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((n, 2, 2, N), dtype=torch.int64, device=device)
    for l in range(2):
        out[:, :, l, :] = torch.randint(0, Q[l], (n, 2, N), generator=g, device=device, dtype=torch.int64)
    return out


def cpu_baseline(a_np, b_np, rk_np, threads: int):
    """Times the oracle (CPU restatement of the SEAL 4.0 path) on a bounded sample. Returns (ops/s, outputs)."""
    from oracle import bfv

    out, secs = bfv.batch_mul_relin(a_np, b_np, rk_np, threads)
    return a_np.shape[0] / secs, out, secs


def e2e_frames(fdev, a_h, b_h, out_h, rk_host, device_index, steps, world, barrier, dist) -> dict:
    """ops/s of fhe_b200_mul_relin_frames on pinned host buffers of structured frames; result frames checked against the
    library's own serialisation of the limb-array result."""
    import ctypes

    import numpy as np
    import torch

    from fhe_precompiles_b200 import _lib
    from fhe_precompiles_b200.sharding import max_over_ranks

    L = _lib.lib()
    dt_ = b"sunscreen::types::bfv::signed::Signed,0.8.1,true"
    fb, fs = fdev.frame_bytes(), fdev.frame_stride()

    def frame_of(words) -> np.ndarray:
        o, ln = ctypes.c_void_p(), ctypes.c_int64()
        w = np.ascontiguousarray(words)
        if L.fhe_b200_write_ciphertext(w.ctypes.data, dt_, ctypes.byref(o), ctypes.byref(ln)) != 0:
            raise RuntimeError("write_ciphertext failed")
        raw = np.frombuffer(ctypes.string_at(o, ln.value), dtype=np.uint8)[ln.value - fb :].copy()  # the zstd frame is the tail
        L.fhe_free(o)
        return raw

    n = a_h.shape[0]
    an, bn = a_h.numpy().view(np.uint64), b_h.numpy().view(np.uint64)
    # this entry point speaks structured frames only (status 1 otherwise); the process default writer is libzstd level 3
    prev_writer = L.fhe_b200_set_zstd_writer(1)
    fa = torch.zeros((n, fs), dtype=torch.uint8).pin_memory()
    fbuf = torch.zeros((n, fs), dtype=torch.uint8).pin_memory()
    for i in range(n):
        fa[i, :fb] = torch.from_numpy(frame_of(an[i]))
        fbuf[i, :fb] = torch.from_numpy(frame_of(bn[i]))
    fo = torch.zeros((n, fs), dtype=torch.uint8).pin_memory()
    st = torch.zeros((n,), dtype=torch.int32).pin_memory()
    for _ in range(2):
        fdev.mul_relin_frames(fa, fbuf, rk_host, fo, st, device=device_index)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        fdev.mul_relin_frames(fa, fbuf, rk_host, fo, st, device=device_index)
    dt = time.perf_counter() - t0
    barrier()
    dt_max = max_over_ranks(dt, dist)
    on = out_h.numpy().view(np.uint64)
    same = all(bool((fo[i, :fb].numpy() == frame_of(on[i])).all()) for i in (0, 1, n // 2, n - 1))
    L.fhe_b200_set_zstd_writer(prev_writer)
    ok = bool((st == 0).all())
    if not (ok and same):  # a rate over rejected frames is not a measurement
        raise RuntimeError(f"fhe_b200_mul_relin_frames: statuses ok={ok}, frames match the limb-array result={same}")
    return {
        "value": world * n * steps / dt_max,
        "unit": "ops/s",
        "h2d_bytes_per_step": 2 * n * fs + rk_host.numel() * 8,
        "d2h_bytes_per_step": n * fs + 12 * n,
        "api": "fhe_b200_mul_relin_frames (C ABI, pinned host buffers of structured zstd frames, 82,054 bytes per ciphertext)",
        "all_status_ok": ok,
        "frames_match_limb_array_result": same,
    }


def e2e_byte_surface(fdev, a, b, net_pub: bytes, steps: int, world: int, barrier, dist, n_calls: int = 4096, distinct: int = 512) -> dict:
    """The metric through the reference's TRUE byte surface: `n_calls` packed mul_cipheri64_cipheri64 inputs (pack.rs framing:
    offsets + the 411 KB PublicKey + two bincode ciphertexts whose SEAL blobs are libzstd level-3 frames, as SEAL writes them)
    in ordinary host memory -> fhe_b200_batch -> packed result bytes in malloc'd buffers.  Everything the reference does per
    call is inside the timed region: framing, key lookup, operand inflate + validation, H2D, kernels, D2H, result framing."""
    import ctypes

    import numpy as np

    from fhe_precompiles_b200 import FHE, _lib, pack
    from fhe_precompiles_b200.sharding import max_over_ranks

    L = _lib.lib()
    dt_ = b"sunscreen::types::bfv::signed::Signed,0.8.1,true"

    def to_bytes(words) -> bytes:
        o, ln = ctypes.c_void_p(), ctypes.c_int64()
        w = np.ascontiguousarray(words)
        assert L.fhe_b200_write_ciphertext(w.ctypes.data, dt_, ctypes.byref(o), ctypes.byref(ln)) == 0
        buf = ctypes.string_at(o.value, ln.value)
        L.fhe_free(o)
        return buf

    an, bn = a[:distinct].cpu().numpy().view(np.uint64), b[:distinct].cpu().numpy().view(np.uint64)
    prev = L.fhe_b200_set_zstd_writer(0)  # operands as SEAL writes them: libzstd level 3
    packed = [pack.pack_binary_operation(net_pub, to_bytes(an[i]), to_bytes(bn[i])) for i in range(distinct)]
    L.fhe_b200_set_zstd_writer(prev)
    bufs = [(ctypes.c_char * len(p)).from_buffer_copy(p) for p in packed]  # every call has its own copy of the key bytes
    op_index = L.fhe_b200_op_index(b"mul_cipheri64_cipheri64")
    arr = (_lib.BatchCall * n_calls)()
    in_bytes = 0
    for i in range(n_calls):
        arr[i].op, arr[i].bytes, arr[i].bytes_length = op_index, ctypes.cast(bufs[i % distinct], ctypes.c_void_p), len(packed[i % distinct])
        in_bytes += len(packed[i % distinct])
    threads = max(2, 2 * (os.cpu_count() or 2) // world)

    def one_batch(check: bool = False, arr=arr, n_calls=n_calls) -> int:
        failed = L.fhe_b200_batch(arr, n_calls, threads)
        out_bytes = 0
        first = ctypes.string_at(arr[0].output, arr[0].output_length) if check and arr[0].status == 0 else None
        for i in range(n_calls):
            out_bytes += arr[i].output_length
            L.fhe_free(arr[i].output)
        if check:
            assert failed == 0 and first == FHE.mul_cipheri64_cipheri64(packed[0])
        return out_bytes

    def timed(mode: int) -> tuple:
        prev_ = L.fhe_b200_set_zstd_writer(mode)
        try:
            out_bytes_ = one_batch(check=True)  # warm (lanes grow to their tile size) + result check against the single-call symbol
            one_batch()
            barrier()
            reps = max(2, min(steps, 5))
            t0 = time.perf_counter()
            for _ in range(reps):
                one_batch()
            dt = time.perf_counter() - t0
            barrier()
            return world * n_calls * reps / max_over_ranks(dt, dist), out_bytes_
        finally:
            L.fhe_b200_set_zstd_writer(prev_)

    rate_seal, out_seal = timed(0)
    rate_struct, out_struct = timed(1)
    # a larger batch with the structured writer: the device zstd decoder's rate grows with the frames per launch (one rank only:
    # with several ranks on one host the leg is host-bound either way and its pinned lanes would only add warm-up time)
    big_n, rate_big = 4 * n_calls, None
    if world == 1:
        big = (_lib.BatchCall * big_n)()
        for i in range(big_n):
            big[i].op, big[i].bytes, big[i].bytes_length = op_index, ctypes.cast(bufs[i % distinct], ctypes.c_void_p), len(packed[i % distinct])
        prev_ = L.fhe_b200_set_zstd_writer(1)
        try:
            one_batch(check=True, arr=big, n_calls=big_n)
            one_batch(arr=big, n_calls=big_n)
            t0 = time.perf_counter()
            for _ in range(3):
                one_batch(arr=big, n_calls=big_n)
            rate_big = big_n * 3 / (time.perf_counter() - t0)
        finally:
            L.fhe_b200_set_zstd_writer(prev_)
    return {
        "value": rate_seal,
        "unit": "calls/s",
        "calls_per_step": n_calls,
        "distinct_inputs": distinct,
        "host_threads": threads,
        "input_bytes_per_step": in_bytes,
        "output_bytes_per_step": out_seal,
        "api": "fhe_b200_batch over pack.rs-framed inputs (c_fhe_mul_cipheri64_cipheri64 semantics per call); operand frames libzstd "
               "level 3; results written with libzstd level 3 on the host pool = byte for byte what SEAL's save() writes (default)",
        "structured_writer": {"value": rate_struct, "unit": "calls/s", "output_bytes_per_step": out_struct,
                              "note": "fhe_b200_set_zstd_writer(1): result frames laid out directly, written on the GPU",
                              "calls_per_s_at_%d_calls" % big_n: rate_big},
        "device_zstd": os.environ.get("FHE_B200_DEVICE_ZSTD", "default") + " (default 2: a batch of >= 2,048 calls runs as big tiles - an eighth of "
                       "the batch, 256..1,024 calls - whose libzstd operand frames are inflated on the GPU: k_zd2_parse / k_zd3_seq / "
                       "k_zd3_exec, byte-identical to libzstd or handed back; 0: host libzstd only)",
    }


def pcie_ceiling(torch, dev, world: int, barrier, dist, seconds: float = 0.6) -> dict:
    """Platform ceiling of the host-buffer paths: pinned-memory H2D and D2H cudaMemcpyAsync running concurrently on two streams
    (64 MiB per copy, like one pipeline chunk), every rank at once; whole-job GB/s = sum over ranks."""
    from fhe_precompiles_b200.sharding import max_over_ranks

    nbytes = 64 << 20
    h_in = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d_in = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_out = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    half = nbytes // 2

    def run(both, h2d: bool, iters: int):
        for _ in range(iters):
            if both or h2d:
                with torch.cuda.stream(s1):
                    d_in.copy_(h_in, non_blocking=True)
            if both == "2to1":  # the workload's byte ratio: two operands in for one result out
                with torch.cuda.stream(s2):
                    h_out[:half].copy_(d_out[:half], non_blocking=True)
            elif both or not h2d:
                with torch.cuda.stream(s2):
                    h_out.copy_(d_out, non_blocking=True)
        s1.synchronize(), s2.synchronize()

    res = {}
    # "h2d_with_half_d2h": H2D GB/s while D2H moves half as many bytes concurrently -- the ratio of both host-buffer paths
    # (two operands in, one result out), so the ceiling that applies to them
    for name, both, h2d in (("h2d_alone", False, True), ("d2h_alone", False, False), ("concurrent", True, True),
                            ("h2d_with_half_d2h", "2to1", True)):
        run(both, h2d, 4)
        iters = 16
        while True:  # calibrate: one burst must last >= seconds / 4 (dt_max is global, so every rank takes the same branch)
            barrier()
            t0 = time.perf_counter()
            run(both, h2d, iters)
            dt_max = max_over_ranks(time.perf_counter() - t0, dist)
            if dt_max >= seconds / 4 or iters >= 4096:
                break
            iters = min(4096, int(iters * max(2.0, seconds / 4 / max(dt_max, 1e-4))))
        best = world * iters * nbytes / dt_max / 1e9
        for rep in range(3):  # best of four timed bursts: a ceiling, not an average
            barrier()
            t0 = time.perf_counter()
            run(both, h2d, iters)
            dt_max = max_over_ranks(time.perf_counter() - t0, dist)
            best = max(best, world * iters * nbytes / dt_max / 1e9)
        res[name + "_GBps_per_direction"] = best
    return res


def call_latency(fdev, a, b, device_index: int, net_pub: bytes, calls: int = 1000) -> dict:
    """p50 / p99 of one c_fhe_mul_cipheri64_cipheri64 call (warm key cache): packed bytes in, packed bytes out,
    i.e. bincode + zstd inflate of two ciphertexts, H2D, six kernels, D2H, zstd deflate.  Also times the codec alone."""
    import ctypes

    import numpy as np

    from fhe_precompiles_b200 import FHE, _lib, pack

    L = _lib.lib()
    dt = b"sunscreen::types::bfv::signed::Signed,0.8.1,true"

    def to_bytes(t):
        w = t.cpu().numpy().view(np.uint64).copy()
        out, n = ctypes.c_void_p(), ctypes.c_int64()
        assert L.fhe_b200_write_ciphertext(w.ctypes.data, dt, ctypes.byref(out), ctypes.byref(n)) == 0
        buf = ctypes.string_at(out.value, n.value)
        L.fhe_free(out)
        return buf

    # operands as the reference's SEAL writes them (libzstd level-3 frames).  Measured under both result writers: "seal"
    # (default: libzstd level 3 on the host, byte-identical to SEAL's save()) and "structured" (frames laid out directly,
    # written on the GPU); `chained` = operands that are themselves structured frames.
    prev = L.fhe_b200_set_zstd_writer(0)
    ca, cb = to_bytes(a[0]), to_bytes(b[0])
    L.fhe_b200_set_zstd_writer(1)
    packed_chained = pack.pack_binary_operation(net_pub, to_bytes(a[0]), to_bytes(b[0]))
    L.fhe_b200_set_zstd_writer(prev)
    packed = pack.pack_binary_operation(net_pub, ca, cb)
    nb = 2048
    op_index = L.fhe_b200_op_index(b"mul_cipheri64_cipheri64")

    def batch_rate(src_bytes):
        # throughput of the same call through fhe_b200_batch (tiles of calls per lane, codec on all host threads); only the C
        # call is timed -- building the call array and copying the outputs into Python objects is the harness, not the library
        src = (ctypes.c_char * len(src_bytes)).from_buffer_copy(src_bytes)
        arr = (_lib.BatchCall * nb)()
        best, first = 0.0, None
        for rep in range(4):  # first repetition warms the lanes (each grows its staging to a tile)
            for i in range(nb):
                arr[i].op, arr[i].bytes, arr[i].bytes_length = op_index, ctypes.cast(src, ctypes.c_void_p), len(src_bytes)
            t0 = time.perf_counter()
            failed = L.fhe_b200_batch(arr, nb, 0)
            dt_ = time.perf_counter() - t0
            assert failed == 0
            first = ctypes.string_at(arr[0].output, arr[0].output_length)
            for i in range(nb):
                L.fhe_free(arr[i].output)
            if rep:
                best = max(best, nb / dt_)
        return best, first

    def p50_p99(data, n):
        for _ in range(5):
            out_ = FHE.mul_cipheri64_cipheri64(data)
        ts = []
        for _ in range(n):
            t0 = time.perf_counter()
            out_ = FHE.mul_cipheri64_cipheri64(data)
            ts.append(time.perf_counter() - t0)
        ts.sort()
        return ts[len(ts) // 2] * 1e3, ts[min(len(ts) - 1, int(len(ts) * 0.99))] * 1e3, out_

    def under(mode: int) -> dict:
        prev_ = L.fhe_b200_set_zstd_writer(mode)
        try:
            p50, p99, out = p50_p99(packed, calls)
            # phase split of the same call (SURVEY 8d): host clock around the codec phases, CUDA events on the lane's stream
            L.fhe_b200_set_call_timing(1)
            phases = ("unpack_key", "parse_inflate", "h2d", "kernels", "d2h", "deflate", "total")
            rows = []
            us = (ctypes.c_double * 7)()
            for _ in range(calls):
                FHE.mul_cipheri64_cipheri64(packed)
                L.fhe_b200_last_call_breakdown(us)
                rows.append(list(us))
            L.fhe_b200_set_call_timing(0)
            split = {f"{k}_us": sorted(r[i] for r in rows)[len(rows) // 2] for i, k in enumerate(phases)}
            # codec alone: inflate both operands + deflate one result, same thread
            words = np.zeros(4 * N, dtype=np.uint64)
            name = ctypes.create_string_buffer(128)
            cs = []
            for _ in range(50):
                t0 = time.perf_counter()
                L.fhe_b200_parse_ciphertext(ca, len(ca), words.ctypes.data, name, 128)
                L.fhe_b200_parse_ciphertext(cb, len(cb), words.ctypes.data, name, 128)
                o, n = ctypes.c_void_p(), ctypes.c_int64()
                L.fhe_b200_write_ciphertext(words.ctypes.data, dt, ctypes.byref(o), ctypes.byref(n))
                L.fhe_free(o)
                cs.append(time.perf_counter() - t0)
            cs.sort()
            rate, first = batch_rate(packed)
            assert first == out
            res = {"p50_ms": p50, "p99_ms": p99, "p50_split": split, "codec_only_p50_ms": cs[len(cs) // 2] * 1e3,
                   "output_bytes": len(out), "batch_calls_per_s": rate}
            if mode == 1:
                res["chained_p50_ms"] = p50_p99(packed_chained, calls)[0]
                res["chained_batch_calls_per_s"] = batch_rate(packed_chained)[0]
            return res
        finally:
            L.fhe_b200_set_zstd_writer(prev_)

    seal, structured = under(0), under(1)
    return {
        "api": "c_fhe_mul_cipheri64_cipheri64 (packed bytes in/out, warm key cache); operand frames libzstd level 3 (as SEAL writes them)",
        "calls": calls,
        "p50_ms": seal["p50_ms"],
        "p99_ms": seal["p99_ms"],
        "p50_split": seal["p50_split"],
        "codec_only_p50_ms": seal["codec_only_p50_ms"],
        "input_bytes": len(packed),
        "output_bytes": seal["output_bytes"],
        "result_writer": "libzstd level 3 on the host (default): result bytes identical to SEAL's save()",
        "byte_surface_batch": {"calls": nb, "calls_per_s": seal["batch_calls_per_s"], "host_threads": os.cpu_count(),
                               "api": "fhe_b200_batch (packed bytes; 2,048 calls: big tiles of 256, operand frames inflated on the GPU)"},
        "structured_writer": dict(structured, note="fhe_b200_set_zstd_writer(1): result frames laid out directly (82,202 bytes), written "
                                                   "on the GPU; chained_* = operands that are such frames too"),
    }


# ---- the reference's byte-surface call on the CPU (fhe.rs:21-30 + pack.rs:238-266), restated with the format oracle:
# deserialise the PublicKey (two zstd blobs), both ciphertext operands, multiply + relinearise, serialise the result with
# zstd level 3.  Forked workers (one per host core) share the packed inputs through the parent's address space.
_BS_CALLS = None


def _bs_worker(rng_):
    from oracle import bfv
    from oracle import formats as F

    from fhe_precompiles_b200 import pack  # pure-Python mirror of pack.rs (no GPU, no library call)

    lo, hi = rng_
    total = 0
    for i in range(lo, hi):
        pkb, ab, bb = pack.unpack_binary_operation(_BS_CALLS[i])
        rk = bfv.rk_array(F.PublicKey.from_bytes(pkb).relin())
        a, b = F.Ciphertext.from_bytes(ab), F.Ciphertext.from_bytes(bb)
        out = bfv.mul_relin(a.polys(), b.polys(), rk)
        total += len(F.make_ciphertext("i64", out).to_bytes())
    return total


def cpu_byte_surface(calls, cores: int, reps: int = 1):
    """calls/s of the CPU byte-surface path over `calls` (list of packed inputs) on `cores` forked workers."""
    import multiprocessing as mp

    global _BS_CALLS
    _BS_CALLS = calls
    n = len(calls)
    step = (n + cores - 1) // cores
    ranges = [(lo, min(n, lo + step)) for lo in range(0, n, step)]
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(_bs_worker, [(0, 1)] * cores)  # warm: imports, liboracle, libzstd in every worker
        t0 = time.perf_counter()
        for _ in range(reps):
            pool.map(_bs_worker, ranges)
        dt = time.perf_counter() - t0
    return n * reps / dt, dt


def oracle_packed_calls(n: int, seed: int, net_pub: bytes):
    """n packed `mul_cipheri64_cipheri64` inputs whose operands are serialised as SEAL writes them (bincode + zstd level 3)."""
    import numpy as np

    from oracle import formats as F

    from fhe_precompiles_b200 import pack

    rng = np.random.default_rng(seed)
    calls = []
    for _ in range(n):
        cts = np.empty((2, 2, 2, N), dtype=np.uint64)
        for l in range(2):
            cts[:, :, l, :] = rng.integers(0, Q[l], size=(2, 2, N), dtype=np.uint64)
        sa, sb = (F.make_ciphertext("i64", c).to_bytes() for c in cts)
        calls.append(pack.pack_binary_operation(net_pub, sa, sb))
    return calls


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np

    from oracle import bfv
    from oracle import formats as F

    cores = os.cpu_count() or 1
    rng = np.random.default_rng(2)
    sample = args.batch  # the SAME batch as the b200 arm: 4,096 ct x ct multiply + relinearise per step
    a = np.empty((sample, 2, 2, N), dtype=np.uint64)
    b = np.empty_like(a)
    for l in range(2):
        a[:, :, l, :] = rng.integers(0, Q[l], size=(sample, 2, N), dtype=np.uint64)
        b[:, :, l, :] = rng.integers(0, Q[l], size=(sample, 2, N), dtype=np.uint64)
    net_pub = open(os.path.join(ROOT, "fhe_precompiles_b200/data/network.pub"), "rb").read()
    pk = F.PublicKey.from_bytes(net_pub)
    rk = bfv.rk_array(pk.relin())
    for _ in range(args.warmup):
        bfv.batch_mul_relin(a, b, rk, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out, _ = bfv.batch_mul_relin(a, b, rk, cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, sample, lambda rows: out[rows])
    value = sample * args.steps / dt
    # the same op through the reference's BYTE surface on the CPU (packed bytes in, packed bytes out), bounded sample
    bs = None
    if not args.no_e2e:
        n_bs = max(8 * cores, 128)
        calls = oracle_packed_calls(n_bs, 5, net_pub)
        rate, secs = cpu_byte_surface(calls, cores, reps=4)
        bs = {"value": rate, "unit": "calls/s", "cores": cores, "sample": f"4 x {n_bs} packed mul_cipheri64_cipheri64 calls, {secs:.2f} s",
              "what": "PublicKey + 2 operands inflated (libzstd), oracle multiply + relinearise, result deflated at zstd level 3, per call"}
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": "ops/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "u64",
        "data": "synthetic uniform residues mod (q0,q1), seed 2",
        "config": {"workload": WORKLOAD, "ops_per_gpu_per_step": sample, "same_config": sample == 4096,
                   "note": "one step = the whole 4,096-op batch on every host thread (limb arrays in host memory, like the b200 arm's e2e)"},
        "cpu_baseline": {
            "value": value,
            "unit": "ops/s",
            "cores": cores,
            "kind": "port",
            "sample": f"{sample} ct*ct multiply+relin per step on {cores} host threads; the reference's SEAL-backed "
            "path cannot be built here (no Rust toolchain, SEAL un-vendored), so this is the C restatement in oracle/",
        },
        "e2e": {"value": value, "unit": "ops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if bs is not None:
        line["byte_surface"] = bs
    print(json.dumps(line), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="ct x ct ops per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the quick runs of BASELINE configs 2, 4 and 5")
    ap.add_argument("--sustain-seconds", type=float, default=0.0, help="extra device-resident run of at least this long with the clock sampler (recorded under `sustained`)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="ops in the CPU-baseline sample (0 = ~20 s of CPU work)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a fixed sample of the last step's results "
                    "to DIR/*.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bind_to_gpu_numa_node(local_rank)
    dist = None
    if world > 1:
        # plumbing only: a barrier and the max-over-ranks of the timing. The path has no data exchange between GPUs,
        # so no NCCL communicator is created (gloo over loopback carries the two scalars).
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime

        dist.init_process_group("gloo", timeout=datetime.timedelta(seconds=600))  # a lost rank fails the run instead of hanging it

    os.environ.setdefault("FHE_B200_DEVICES", str(local_rank))  # this rank's byte-surface calls stay on its own GPU
    from fhe_precompiles_b200 import device as fdev

    fdev.init(local_rank)
    n = args.batch
    a = synth_ciphertexts(torch, n, 2 + 2 * rank, dev)
    b = synth_ciphertexts(torch, n, 3 + 2 * rank, dev)
    out = torch.empty_like(a)
    net_pub = open(os.path.join(ROOT, "fhe_precompiles_b200/data/network.pub"), "rb").read()
    _, rk_host = fdev.parse_public_key(net_pub)
    rk = rk_host.to(dev)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------- device-resident timed region
    for _ in range(args.warmup):
        fdev.mul_relin(a, b, rk, out=out)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    fdev.set_kernel_timing(True)
    launches0 = fdev.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        fdev.mul_relin(a, b, rk, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = fdev.launch_count() - launches0
    kt = fdev.kernel_timing_report(local_rank)
    fdev.set_kernel_timing(False)
    clocks = sampler.stop()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, n, lambda rows: out[torch.from_numpy(rows).to(dev)].cpu().numpy().view(np.uint64))
    from fhe_precompiles_b200.sharding import max_over_ranks, whole_job_rate

    ms_max = max_over_ranks(ms, dist)
    value = whole_job_rate(n * args.steps, world, ms_max * 1e-3)

    # ---------------- optional sustained run (>= --sustain-seconds of back-to-back steps): clocks, power and rate under a long load
    sustained = None
    if args.sustain_seconds > 0:
        sampler2 = ClockSampler(local_rank)
        sampler2.start()
        steps_s = 0
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall = time.perf_counter()
        s0.record()
        while time.perf_counter() - t_wall < args.sustain_seconds:
            for _ in range(25):
                fdev.mul_relin(a, b, rk, out=out)
            steps_s += 25
            torch.cuda.synchronize()
        s1.record()
        torch.cuda.synchronize()
        ms_s = s0.elapsed_time(s1)
        sustained = {"seconds": ms_s * 1e-3, "steps": steps_s, "ops_per_s_per_gpu": n * steps_s / (ms_s * 1e-3), "clocks": sampler2.stop(),
                     "ratio_to_timed_region": (n * steps_s / ms_s) / (n * args.steps / ms)}
        barrier()

    # ---------------- end to end through the C ABI with host buffers
    e2e = None
    if not args.no_e2e:
        a_h = a.cpu().pin_memory()
        b_h = b.cpu().pin_memory()
        out_h = torch.empty_like(a_h).pin_memory()
        for _ in range(2):
            fdev.mul_relin_host(a_h, b_h, rk_host, out_h, device=local_rank)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fdev.mul_relin_host(a_h, b_h, rk_host, out_h, device=local_rank)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        dt_max = max_over_ranks(dt, dist)
        same = bool(torch.equal(out_h, out.cpu()))
        e2e = {
            "value": world * n * args.steps / dt_max,
            "unit": "ops/s",
            "h2d_bytes_per_step": 2 * n * CT_BYTES + rk_host.numel() * 8,
            "d2h_bytes_per_step": n * CT_BYTES,
            "api": "fhe_b200_mul_relin_host (C ABI, pinned host limb arrays)",
            "matches_device_resident_result": same,
        }
        # the same batch with SERIALIZED operands: structured zstd frames (5 bytes per residue, what this library's precompiles
        # return and accept) in and out through fhe_b200_mul_relin_frames; frames are unpacked / written on the GPU
        try:
            e2e["serialized"] = e2e_frames(fdev, a_h, b_h, out_h, rk_host, local_rank, args.steps, world, barrier, dist)
        except Exception as ex:  # pragma: no cover
            e2e["serialized"] = {"error": str(ex)}
        del a_h, b_h, out_h
        # the platform's ceiling for those two paths: concurrent pinned H2D + D2H on every rank at once
        try:
            ceil = pcie_ceiling(torch, dev, world, barrier, dist)
            h2d_rate = ceil["h2d_with_half_d2h_GBps_per_direction"] * 1e9  # both paths move 2 bytes in per byte out
            lim = lambda h2d, d2h: min(h2d_rate / (h2d / n), h2d_rate / 2 / (d2h / n))  # ops/s if the copies were all there is
            ceil["limb_arrays_ops_per_s"] = lim(e2e["h2d_bytes_per_step"], e2e["d2h_bytes_per_step"])
            e2e["frac_of_platform_ceiling"] = e2e["value"] / ceil["limb_arrays_ops_per_s"]
            if "value" in e2e["serialized"]:
                ceil["frames_ops_per_s"] = lim(e2e["serialized"]["h2d_bytes_per_step"], e2e["serialized"]["d2h_bytes_per_step"])
                e2e["serialized"]["frac_of_platform_ceiling"] = e2e["serialized"]["value"] / ceil["frames_ops_per_s"]
            if e2e["frac_of_platform_ceiling"] > 1.0:
                ceil["note"] = ("the copy-only bursts ran slower than the pipeline's sustained copies: with several ranks on one host "
                                "the pinned-memory rate is set by host memory contention and varies between bursts; read the "
                                "fraction as 'at the platform's limit', not as a number above 1")
            e2e["platform_ceiling"] = ceil
        except Exception as ex:  # pragma: no cover
            e2e["platform_ceiling"] = {"error": str(ex)}
        # the reference's true byte surface (packed bytes with libzstd-written operands in, packed bytes out)
        try:
            e2e["byte_surface"] = e2e_byte_surface(fdev, a, b, net_pub, args.steps, world, barrier, dist)
        except Exception as ex:  # pragma: no cover
            e2e["byte_surface"] = {"error": str(ex)}

    # ---------------- the other BASELINE configs (2: NTT microbenchmark, 4: 65,536 mixed calls, 5: 16,384 encrypt + decrypt),
    # sharded over the ranks like the headline (no collective); quick settings, the full sweep is scripts/bench_configs.py
    configs = None
    if not args.no_configs:
        try:
            sys.path.insert(0, os.path.join(ROOT, "scripts"))
            import bench_configs

            configs = bench_configs.run_configs(rank, world, dist, quick=True)
        except Exception as ex:  # pragma: no cover
            configs = {"error": str(ex)}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---------------- single-call latency through the reference's byte surface (metric: "p50 call latency")
    latency = None
    if not args.no_e2e:
        latency = call_latency(fdev, a, b, local_rank, net_pub)

    # ---------------- roofline of the dominant kernel (live CUDA-event durations from the timed region)
    # bound = the 32-bit integer multiplier (FMA-heavy pipe), not HBM: SURVEY 8(d).  achieved = ALGORITHMIC IMAD.WIDE-equivalents
    # per launch of the dominant kernel / its average launch duration; peak = the mul.wide.u32 rate measured on this GPU right
    # here (fhe_b200_int_peak; MEASURED_PEAKS.json holds no integer figure), with the theoretical 148 SM x 32 / clk next to it.
    peak_gbs, peak_src = measured_peaks()
    dom = max(kt, key=lambda k: kt[k][0])
    dom_ms, dom_launches = kt[dom]
    total_kernel_ms = sum(v[0] for v in kt.values())
    ops_per_launch = n * args.steps / max(dom_launches, 1)
    avg_launch_ms = dom_ms / max(dom_launches, 1)
    prof = {}
    try:  # the committed ncu capture (profiles/): DRAM bytes per op and FMA-heavy pipe utilisation of each kernel
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            prof = json.load(f)
    except Exception:
        prof = {}
    def slot_of(ncu_kernel: str) -> str:
        """timed slot of an ncu kernel name: k_ext_ntt2 / k_ext_ntt_d<0> -> k_ext_ntt, k_ks_finish<1> -> k_ks_finish, ..."""
        k = ncu_kernel.split("<")[0]
        if k.endswith("_ksd") or k == "k_tensor_floor_d":
            return k
        if k.endswith("_d"):
            k = k[:-2]
        return "k_ext_ntt" if k == "k_ext_ntt2" else k

    table = {slot_of(k): v for k, v in prof.get("dram_bytes_per_op", {}).items()}
    heavy = {slot_of(k): v for k, v in (prof.get("fmaheavy_pct") or {}).items()}
    traffic = table[dom] * ops_per_launch if dom in table else None
    sm_clock_ghz = (clocks.get("sm_mhz") or 1965.0) / 1e3
    peak_theory = SM_COUNT * WIDE_PER_CLK_PER_SM * sm_clock_ghz / 1e3  # T IMAD.WIDE/s at the clock observed under load
    try:
        peak_wide = fdev.int_peak(local_rank, wide=1)  # T IMAD.WIDE/s (mul.wide.u32 with a loop-carried operand)
        peak_lo = fdev.int_peak(local_rank, wide=0)
        bf_small, bf_big = fdev.bfly_peak(local_rank, 0), fdev.bfly_peak(local_rank, 3)
    except Exception as e:  # pragma: no cover
        raise SystemExit(f"bench.py: integer-pipe probe failed: {e}")
    ops_s = n * args.steps / (ms * 1e-3)
    dom_weq = KERNEL_WIDE_EQ.get(dom)
    ach_dom = dom_weq * ops_per_launch / (avg_launch_ms * 1e-3) / 1e12 if dom_weq else None
    ach_op = ops_s * WIDE_EQ_PER_OP / 1e12
    per_kernel = {}
    for k, (kms, kl) in kt.items():
        if k in KERNEL_WIDE_EQ and kms > 0:
            ach_k = KERNEL_WIDE_EQ[k] * n * args.steps / (kms * 1e-3) / 1e12
            per_kernel[k] = {"us_per_op": kms * 1e3 / (n * args.steps), "achieved": ach_k, "frac": ach_k / peak_wide,
                             "frac_of_theoretical": ach_k / peak_theory,
                             "share_of_step": kms / total_kernel_ms,
                             "ncu_fmaheavy_pct": heavy.get(k)}
    ntt_floor_us = 24576 * ((26 if QLIMB_NTT else 12) / bf_small + 21 / bf_big) * 1e-3  # 64-bit-lane butterfly rates (SEAL's primes)
    hbm_ach = ops_per_launch * ALGO_BYTES_PER_OP / (avg_launch_ms * 1e-3) / 1e9
    roofline = {
        "bound": "int_pipe",
        "kernel": dom,
        "achieved": ach_dom,
        "peak": peak_wide,
        "unit": "T IMAD.WIDE-equivalents/s (32-bit multiplier, FMA-heavy pipe)",
        "frac": ach_dom / peak_wide if ach_dom else None,
        "traffic": traffic,
        "peak_source": "measured here: fhe_b200_int_peak (mul.wide.u32, loop-carried operands, 2 x 1024 threads per SM)",
        "peak_theoretical": peak_theory,
        "frac_of_theoretical": ach_dom / peak_theory if ach_dom else None,
        "algorithmic_wide_eq_per_op": {"dominant_kernel": dom_weq, "whole_op": WIDE_EQ_PER_OP,
                                       "limb_ntts_per_op": NTTS_PER_OP,
                                       "behz": BEHZ,
                                       "key_switch": KS,
                                       "model": {"seal": "SEAL's form, 14+12 fwd / 12+9 inv limb-NTTs",
                                                 "bsk": "q-limbs of the tensor product recovered from its Bsk limbs: 6+12 fwd / 6+9 inv limb-NTTs",
                                                 "dual": "tensor product on six primes below 2^30, two per word: 12 fwd + 9 inv dual transforms at 4.0 "
                                                         "IMAD.WIDE-equivalents per butterfly (both lanes), 6 fwd + 6 inv key-switch transforms (dual too "
                                                         "unless FHE_B200_KS=seal)"}[BEHZ]
                                                + " x 24,576 butterflies at 6.5 / 7.0 (36-37 bit) and 7.5 (61 bit) "
                                                "IMAD.WIDE-equivalents + pointwise per kernel (bench.py KERNEL_WIDE_EQ, DESIGN.md section 4)"},
        "whole_op": {"achieved": ach_op, "frac": ach_op / peak_wide, "frac_of_theoretical": ach_op / peak_theory, "us_per_op": 1e6 / ops_s,
                     "pipe_bound_us_per_op": WIDE_EQ_PER_OP / (peak_wide * 1e12) * 1e6},
        "per_kernel": per_kernel,
        "avg_launch_ms": avg_launch_ms,
        "ops_per_launch": ops_per_launch,
        "kernel_share_of_step": dom_ms / total_kernel_ms if total_kernel_ms else None,
        "measured_pipe_rates_T_per_s": {"IMAD.WIDE": peak_wide, "IMAD": peak_lo},
        "butterfly_peak_G_per_s": {"36-37 bit primes": bf_small, "61 bit primes": bf_big},
        "ntt_only_floor_us_per_op": ntt_floor_us,
        "ncu": {"tag": prof.get("tag"), "fmaheavy_pct": prof.get("fmaheavy_pct")},
        # secondary: the HBM form SURVEY 8(d) defines (393,216 algorithmic bytes per op) -- the op is far from HBM-bound
        "hbm": {
            "achieved": hbm_ach, "peak": peak_gbs, "unit": "GB/s", "frac": hbm_ach / peak_gbs, "peak_source": peak_src,
            "algorithmic_bytes_per_op": ALGO_BYTES_PER_OP,
            "whole_op_frac": ops_s * ALGO_BYTES_PER_OP / 1e9 / peak_gbs,
            "dram_bytes_per_op_ncu": prof.get("dram_bytes_per_op_total"),
            "traffic_over_algorithmic": (prof.get("dram_bytes_per_op_total") or 0) / ALGO_BYTES_PER_OP or None,
        },
    }

    line = {
        "metric": METRIC,
        "value": value,
        "unit": "ops/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "u64",
        "data": "synthetic uniform residues mod (q0,q1), seed 2",
        "config": {
            "workload": WORKLOAD,
            "ops_per_gpu_per_step": n,
            "l2": "inputs (1 GiB per GPU) exceed the 126 MB L2; no flush needed",
            "sharding": f"{world} rank(s), independent batches, no collective",
            "chunk_ops": int(os.environ.get("FHE_B200_CHUNK_OPS", "4096")),
            "subchunk_ops": int(os.environ.get("FHE_B200_SUBCHUNK_OPS", "0")),
            "kernels": ("multi-polynomial CTAs (FHE_B200_FUSED)" if int(os.environ.get("FHE_B200_FUSED", "0")) else
                        f"one polynomial per CTA; BEHZ base {BEHZ}, key switch {KS}, fused tails {FUSE_TAIL}"),
        },
        "roofline": roofline,
        "clocks": clocks,
        "gpu_launches": int(launches),
    }
    if e2e is not None:
        line["e2e"] = e2e
    if latency is not None:
        line["latency"] = latency
    if configs is not None:
        line["configs"] = configs
    if sustained is not None:
        line["sustained"] = sustained

    # ---------------- CPU baseline on the box's host cores (N=1 only), also the parity checker for the sample
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        sample = args.cpu_sample or min(n, max(64, int(20.0 / 0.010)))  # ~20 s of single-core work at ~10 ms/op
        a_np = a[:sample].cpu().numpy().view(np.uint64)
        b_np = b[:sample].cpu().numpy().view(np.uint64)
        rk_np = rk_host.numpy().view(np.uint64)
        cpu_ops, cpu_out, secs = cpu_baseline(a_np, b_np, rk_np, cores)
        one = []
        for i in range(5):
            _, _, sec1 = cpu_baseline(a_np[i : i + 1], b_np[i : i + 1], rk_np, 1)
            one.append(sec1)
        one.sort()
        # what one call costs the reference on one core THROUGH the byte surface: it deserialises the public key (two zstd
        # blobs), both operands, runs the arithmetic and deflates the result at zstd level 3 (fhe.rs:21-30, pack.rs:238-266)
        from oracle import formats as OF

        z = OF.zstd()
        pkp = OF.PublicKey.from_bytes(net_pub)
        key_blobs = [pkp.public_key.blob[16:], pkp.relin_key.blob[16:]]  # the zstd frames inside the two SEAL blobs
        ct_payload = OF.fresh_data_ciphertext(a_np[0]).payload()
        ct_blob = z.compress(ct_payload, 3)

        def med(fn, reps=9):
            t = []
            for _ in range(reps):
                t0 = time.perf_counter()
                fn()
                t.append(time.perf_counter() - t0)
            return sorted(t)[len(t) // 2] * 1e3

        codec_ms = {
            "inflate_key_ms": med(lambda: [z.decompress(kb) for kb in key_blobs]),
            "inflate_2_operands_ms": med(lambda: [z.decompress(ct_blob), z.decompress(ct_blob)]),
            "deflate_result_ms": med(lambda: z.compress(ct_payload, 3)),
        }
        arith_ms = one[len(one) // 2] * 1e3
        line["cpu_baseline"] = {
            "byte_surface_call_ms_1_thread": {**codec_ms, "arithmetic_ms": arith_ms, "total_ms": arith_ms + sum(codec_ms.values()),
                                              "note": "libzstd calls + oracle arithmetic only; bincode parsing and SEAL context checks not counted"},
            "p50_call_ms_arithmetic_only_1_thread": arith_ms,
            "value": cpu_ops,
            "unit": "ops/s",
            "cores": cores,
            "kind": "port",
            "sample": f"first {sample} ops of the same batch, oracle/ C restatement of the SEAL 4.0 path, {cores} threads, {secs:.2f} s",
            "bit_exact_vs_gpu": bool(np.array_equal(cpu_out, out[:sample].cpu().numpy().view(np.uint64))),
        }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
