"""GPU parity on the crafted boundary operands of tests/edge_inputs.py: every output of every op bit-compared with the oracle,
through each multiply path -- device-resident at both tail forms and a call mixing them, multiply and relinearize alone, the
host-buffer pipeline at every branch of its chunk schedule, the frame pipeline -- and decrypt at the budget thresholds."""
import os
import subprocess
import sys

import numpy as np
import pytest

import edge_inputs as E
from helpers import N, ROOT, random_ct
from oracle import bfv
from oracle import formats as F

pytestmark = pytest.mark.gpu

THREADS = os.cpu_count() or 8
# launches per chunk of the host pipelines (kernels.cu launch_*): fused = ext_conv, ext_ntt, tensor_floor + rk_prepare_ksd (3),
# digit_ntt_ksd, ks_tail_ksd; split = ext_conv, ext_ntt, tensor_intt, floor_sk + digit_ntt, ks_intt, relin_finish
FUSED_LAUNCHES, SPLIT_LAUNCHES = 8, 7


@pytest.fixture(scope="module")
def dev():
    import torch

    from fhe_precompiles_b200 import device

    assert torch.cuda.is_available(), "no CUDA device: the product has no CPU path"
    device.init(0)
    return device


@pytest.fixture(scope="module")
def batch(keys):
    return E.edge_batch(keys.rk)


@pytest.fixture(scope="module")
def want(batch, keys):
    return bfv.batch_mul_relin(batch.a, batch.b, keys.rk, THREADS)[0]


def to_dev(a: np.ndarray):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()


def to_np(t) -> np.ndarray:
    return t.cpu().numpy().view(np.uint64)


def first_bad(got: np.ndarray, want: np.ndarray):
    bad = [i for i in range(len(want)) if not np.array_equal(got[i], want[i])]
    return bad[:10]


def expected_launches(n: int, chunk: int) -> int:
    sched = E.pipe_schedule(n, chunk)
    fused = sum(c >= E.FUSED_TAIL_MIN_OPS for c in sched)
    return FUSED_LAUNCHES * fused + SPLIT_LAUNCHES * (len(sched) - fused)


def test_mul_relin_crafted_at_both_tail_forms(dev, keys, batch, want):
    """the default chunk (one chunk of 256: fused tails, key switch on the dual base), chunks of 64 (split tails, SEAL's key
    primes) and chunks of 100 on 150 ops (100 fused + 50 split in one call); the timing report shows which kernels ran"""
    import torch

    da, db, drk = to_dev(batch.a), to_dev(batch.b), to_dev(keys.rk)
    prev = dev.set_chunk_ops(0)
    fused = {"k_tensor_floor_d", "k_ks_tail_ksd", "k_rk_prepare_ksd", "k_digit_ntt_ksd"}
    split = {"k_tensor_intt", "k_floor_sk", "k_digit_ntt", "k_ks_intt", "k_relin_finish"}
    try:
        for chunk, n, n_fused, n_split in ((4096, 256, 1, 0), (64, 256, 0, 4), (100, 150, 1, 1)):
            dev.set_chunk_ops(chunk)
            dev.set_kernel_timing(True)
            dev.kernel_timing_report()
            out = dev.mul_relin(da[:n].contiguous(), db[:n].contiguous(), drk)
            torch.cuda.synchronize()
            rep = dev.kernel_timing_report()
            dev.set_kernel_timing(False)
            assert {k: rep[k][1] for k in fused if k in rep} == {k: n_fused for k in fused if n_fused}, (chunk, rep)
            assert {k: rep[k][1] for k in split if k in rep} == {k: n_split for k in split if n_split}, (chunk, rep)
            assert rep["k_ext_conv"][1] == n_fused + n_split
            assert first_bad(to_np(out), want[:n]) == [], f"chunk {chunk}"
    finally:
        dev.set_kernel_timing(False)
        dev.set_chunk_ops(prev)


def test_multiply_and_relinearize_crafted(dev, keys, batch):
    """multiply alone against bfv.multiply on every crafted pair, and relinearize alone on the crafted size-3 ciphertexts (U mod
    P on the rounding boundaries, digits at q_j - 1) padded to 128 ops, at the default chunk (fused) and at chunks of 64 (split)"""
    rng = np.random.default_rng(77)
    want3 = np.stack([bfv.multiply(x, y) for x, y in zip(batch.a, batch.b)])
    pad = random_ct(rng, 2 * (128 - len(batch.c3))).reshape(-1, 4, 2, N)[:, :3]
    c3 = np.concatenate([batch.c3, pad])
    want_rl = np.stack([bfv.relinearize(c, keys.rk) for c in c3])
    da, db, dc3, drk = to_dev(batch.a), to_dev(batch.b), to_dev(c3), to_dev(keys.rk)
    prev = dev.set_chunk_ops(0)
    try:
        for chunk in (4096, 64):
            dev.set_chunk_ops(chunk)
            assert first_bad(to_np(dev.multiply(da, db)), want3) == [], f"multiply, chunk {chunk}"
            assert first_bad(to_np(dev.relinearize(dc3, drk)), want_rl) == [], f"relinearize, chunk {chunk}"
    finally:
        dev.set_chunk_ops(prev)


@pytest.fixture(scope="module")
def host_pool(batch, keys):
    """700 ops: the crafted batch, then uniform ops; the oracle's products under both fixture keys"""
    n = max(E.PIPE_NS)
    rng = np.random.default_rng(99)
    a = np.concatenate([batch.a, random_ct(rng, n - len(batch.a))])
    b = np.concatenate([batch.b, random_ct(rng, n - len(batch.b))])
    return a, b, {name: bfv.batch_mul_relin(a, b, rk, THREADS)[0] for name, rk in (("rk", keys.rk), ("net_rk", keys.net_rk))}


def test_mul_relin_host_every_schedule_branch(dev, keys, host_pool):
    """mul_relin_host (the host-buffer pipeline) at n covering every branch of pipe_chunk at its default 256-op chunk, pinned and
    pageable tensors alternating, two consecutive calls with different keys (a stale device key would show in the second);
    launch counts confirm each chunk's tail form, as the mirror of pipe_chunk predicts"""
    import torch

    a, b, want = host_pool
    seen = set()
    for n in E.PIPE_NS:
        E.pipe_schedule(n, 256, seen)
    assert seen == set(E.PIPE_BRANCHES)
    for idx, n in enumerate(E.PIPE_NS):
        pinned = idx % 2 == 0
        host = (lambda t: t.pin_memory()) if pinned else (lambda t: t)
        ta, tb = host(torch.from_numpy(a[:n].view(np.int64))), host(torch.from_numpy(b[:n].view(np.int64)))
        for name in ("rk", "net_rk"):
            rk = torch.from_numpy(getattr(keys, name).view(np.int64))
            out = host(torch.zeros((n, 2, 2, N), dtype=torch.int64))
            before = dev.launch_count()
            dev.mul_relin_host(ta, tb, rk, out)
            assert dev.launch_count() - before == expected_launches(n, 256), (n, E.pipe_schedule(n, 256))
            assert first_bad(out.numpy().view(np.uint64), want[name][:n]) == [], f"n={n} key={name} pinned={pinned}"


_CHILD = r"""
import sys, numpy as np, torch
sys.path.insert(0, sys.argv[1])
from fhe_precompiles_b200 import device
d = sys.argv[2]
a, b, rk = (torch.from_numpy(np.load(f"{d}/{x}.npy").view(np.int64)) for x in ("a", "b", "rk"))
out = torch.zeros_like(a).pin_memory()
device.init(0)
before = device.launch_count()
device.mul_relin_host(a.pin_memory(), b.pin_memory(), rk, out)
print("launches", device.launch_count() - before)
np.save(f"{d}/out.npy", out.numpy().view(np.uint64))
"""


@pytest.mark.parametrize("chunk", [64, 97])
def test_mul_relin_host_pipe_chunk_setting(keys, host_pool, tmp_path, chunk):
    """FHE_B200_PIPE_CHUNK_OPS is read once per device, so each setting runs in its own process: 64 takes pipe_chunk's
    `chunk <= edge` branch (all split), 97 gives 96 / 97 / 11 / 96 on 300 ops (a split chunk between fused ones)"""
    a, b, want = host_pool
    n = 300
    for name, x in (("a", a[:n]), ("b", b[:n]), ("rk", keys.rk)):
        np.save(tmp_path / f"{name}.npy", np.ascontiguousarray(x))
    env = dict(os.environ, FHE_B200_PIPE_CHUNK_OPS=str(chunk))
    r = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(tmp_path)], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert f"launches {expected_launches(n, chunk)}" in r.stdout, (r.stdout, E.pipe_schedule(n, chunk))
    assert first_bad(np.load(tmp_path / "out.npy"), want["rk"][:n]) == []


def test_mul_relin_frames_crafted_mixed_chunks(dev, keys, batch, want):
    """mul_relin_frames on 150 crafted pairs (chunks of 96 fused + 54 split): every result frame equals the format oracle's
    frame of the oracle's product.  Monomials shifted past the first 16 coefficients have no structured frame (the writer
    leaves runs of equal words to libzstd), so those pairs are skipped."""
    import torch

    n = 150
    fb_, fs = dev.frame_bytes(), dev.frame_stride()
    frame = lambda ct: F.zstd_structured_frame(F.fresh_data_ciphertext(ct).payload())
    ops = [i for i in range(len(batch.a)) if frame(batch.a[i]) is not None and frame(batch.b[i]) is not None][:n]
    assert len(ops) == n and sum(batch.kind[i] == "floor" for i in ops) >= 16

    def frames_of(cts):
        buf = np.zeros((n, fs), dtype=np.uint8)
        for r, i in enumerate(ops):
            buf[r, :fb_] = np.frombuffer(frame(cts[i]), dtype=np.uint8)
        return buf

    ta, tb = torch.from_numpy(frames_of(batch.a)).pin_memory(), torch.from_numpy(frames_of(batch.b)).pin_memory()
    out = torch.zeros((n, fs), dtype=torch.uint8).pin_memory()
    status = torch.full((n,), -1, dtype=torch.int32).pin_memory()
    dev.mul_relin_frames(ta, tb, torch.from_numpy(keys.rk.view(np.int64)), out, status)
    assert (status.numpy() == 0).all()
    bad = [i for r, i in enumerate(ops) if out[r, :fb_].numpy().tobytes() != frame(want[i])]
    assert bad == [], bad[:10]


def test_decrypt_at_the_budget_thresholds(dev, keys, batch):
    """decrypt_checked on c1 = 0 ciphertexts whose t X mod q sits at 2^70 - 1, 2^70, q - 2^70, q - 2^70 + 1, (q-1)/2 and (q+1)/2:
    plaintexts equal bfv.decrypt's (ties and near-ties round as the oracle does) and the flag is budget <= 0; through the byte
    surface, decrypt_i64 succeeds at 2^70 - 1 and fails with code 5 at 2^70"""
    from fhe_precompiles_b200 import FHE, FheError, pack

    for sk in (keys.sk, keys.net_sk):
        plain, flags = dev.decrypt_checked(to_dev(batch.dec), to_dev(sk))
        plain, flags = plain.cpu().numpy().view(np.uint16).astype(np.uint64), flags.cpu().tolist()
        for i, ct in enumerate(batch.dec):
            want_plain, budget = bfv.decrypt(ct, sk)
            assert np.array_equal(plain[i], want_plain), batch.dec_classes[i]
            assert flags[i] == int(budget <= 0), (batch.dec_classes[i], budget)
    by_name = {next(iter(c)): ct for c, ct in zip(batch.dec_classes, batch.dec)}
    ser = lambda c: F.make_ciphertext("i64", c).to_bytes()
    ok = by_name["dec:rem=2^70-1"]
    got = pack.deserialize_scalar("i64", FHE.decrypt_i64(ser(ok)))
    assert got == bfv.decode("i64", bfv.decrypt(ok, keys.net_sk)[0])
    with pytest.raises(FheError) as e:
        FHE.decrypt_i64(ser(by_name["dec:rem=2^70"]))
    assert e.value.code == 5
