"""The crafted boundary operands of tests/edge_inputs.py (CPU only): every class is hit, checked with the restated decision
variables; the restatements themselves equal the oracle (which follows SEAL); the dual-base integer formulation equals the
oracle at these edges; the decrypt budget at the crafted thresholds."""
import numpy as np
import pytest

import edge_inputs as E
from helpers import N
from oracle import bfv

M32 = (1 << 32) - 1


@pytest.fixture(scope="module")
def batch(keys):
    return E.edge_batch(keys.rk)


def test_batch_is_mostly_crafted(batch):
    assert len(batch.a) >= 256 and sum(k != "uniform" for k in batch.kind) >= 200


def test_every_class_is_hit(batch, keys):
    """recomputed from the operands, not taken from the generator's bookkeeping"""
    k = E.consts()
    ext = set()
    for i in np.nonzero(np.array(batch.kind) == "ext")[0]:
        got = set().union(*(E.ext_classes(int(x0), int(x1)) for x0, x1 in E._pairs(batch.a[i], batch.b[i])))
        assert batch.classes[i] <= got
        ext |= got
    assert set(E.EXT_CLASSES) <= ext, sorted(set(E.EXT_CLASSES) - ext)

    floor = set()
    for i in np.nonzero(np.array(batch.kind) == "floor")[0]:
        floor |= E.floor_coverage(batch.a[i], batch.b[i])
    assert set(E.FLOOR_CLASSES) <= floor, sorted(set(E.FLOOR_CLASSES) - floor)

    RK = E.rk_integers(keys.rk)
    ks = set()
    for c3, claimed in zip(batch.c3, batch.c3_classes):
        got = set()
        if (c3[2, 0] == k.q0 - 1).all() and (c3[2, 1] == k.q1 - 1).all():
            got.add("ks:digits=q-1")
        else:
            for kk in range(2):
                um = {E.ks_vars(E.ks_U(c3, RK, kk, i))["umodP"] for i in range(N)}
                got |= {f"ks:U%P={n}:k{kk}" for n, tf in E.KS_TARGETS if tf(k.P) in um}
        assert claimed <= got
        ks |= got
    assert set(E.KS_CLASSES) <= ks, sorted(set(E.KS_CLASSES) - ks)

    dec = set()
    for ct, claimed in zip(batch.dec, batch.dec_classes):
        rems = {E.decrypt_vars(x)["rem"] for x in E._ints(ct, 0)}
        got = {f"dec:rem={n}" for n, tf in E.DEC_TARGETS if tf(k.q) in rems}
        assert claimed <= got
        dec |= got
    assert set(E.DEC_CLASSES) <= dec


def test_extension_carry_into_bit_64_cannot_happen():
    """ext_shared's `sAB < A ? 8u : 0u`: A + rm q_w1 stays below 2^64 for every rm < 2^32 and y0 < 2q, with more than 2^54 to
    spare, so the term never fires (and the restatement never sets it on the crafted pool)"""
    k = E.consts()
    A_max = ((2 * k.q - 1) >> 32) + ((M32 * k.q_w[0]) >> 32) + 1
    assert A_max + M32 * k.q_w[1] < (1 << 64) - (1 << 54)


def test_restated_extension_equals_oracle(batch):
    """Z from the restated ext_shared is the integer a' of SEAL's fastbconv_m_tilde + sm_mrq: its residues mod the Bsk primes
    equal the oracle's, on an op built from the crafted pool (every coefficient on a boundary)"""
    k = E.consts()
    q0, q1, P, b0, b1, msk = bfv.moduli()
    i = batch.kind.index("ext")
    ext = bfv.behz_extend(batch.a[i], batch.b[i])  # [4][5][N]
    for p, (ct, poly) in enumerate(((batch.a[i], 0), (batch.a[i], 1), (batch.b[i], 0), (batch.b[i], 1))):
        for c in range(0, N, 7):
            v = E.ext_vars(int(ct[poly, 0, c]), int(ct[poly, 1, c]))
            assert not v["sAB_wrap"]
            assert v["Z"] << 32 == v["y0"] + (v["rm"] - (1 << 32 if v["neg"] else 0)) * k.q
            assert [v["Z"] % m for m in (b0, b1, msk)] == [int(ext[p, e, c]) for e in (2, 3, 4)]


def test_restated_floor_equals_oracle(batch):
    """f = (t D - y0') / q from the restated floor_sk_coeff_d, for every coefficient of the monomial ops at all four shifts and
    both monomial values, equals the oracle's size-3 product"""
    for i in [i for i, kd in enumerate(batch.kind) if kd == "floor"][:8]:
        assert np.array_equal(E.floor_product(batch.a[i], batch.b[i]), bfv.multiply(batch.a[i], batch.b[i])), f"op {i}"


def test_restated_key_switch_equals_oracle(batch, keys):
    """out_l = c_l + (U - (last - P/2)) P^-1 mod q_l from the restated rounded division equals the oracle's relinearisation on
    every crafted size-3 ciphertext with monomial digits"""
    k = E.consts()
    RK = E.rk_integers(keys.rk)
    for c3, cls in zip(batch.c3, batch.c3_classes):
        if "ks:digits=q-1" in cls:
            continue
        want = bfv.relinearize(c3, keys.rk)
        for kk in range(2):
            for i in range(0, N, 3):
                U = E.ks_U(c3, RK, kk, i)
                d = E.ks_vars(U)["last"] - k.half_P
                for l, ql in enumerate((k.q0, k.q1)):
                    assert (int(c3[kk, l, i]) + (U - d) * pow(k.P, -1, ql)) % ql == int(want[kk, l, i])


def test_dual_base_formulation_at_the_edges(batch, keys):
    """scripts/check_dual_base.py's integer formulation (what the kernels run on the six dual primes) equals the oracle on crafted
    pairs: an all-boundary extension op, a wrapped floor op with the largest |A|, a key switch landing on U mod P = (P+1)/2 and
    one with both digits at q_j - 1"""
    m = E._check_dual_base()
    i_ext = batch.kind.index("ext")
    i_floor = next(i for i, kd in enumerate(batch.kind) if kd == "floor" and batch.a[i][0, 0, N - 1]
                   and E._crt(int(batch.a[i][0, 0, N - 1]), int(batch.a[i][0, 1, N - 1])) == (E.consts().q - 1) // 2)
    for i in (i_ext, i_floor):
        assert m.check_multiply(batch.a[i], batch.b[i]) == 0, f"op {i}"
    for c3, cls in zip(batch.c3, batch.c3_classes):
        if cls & {"ks:U%P=(P+1)/2:k0", "ks:digits=q-1"}:
            assert m.check_key_switch(c3, keys.rk) == 0, cls


def test_decrypt_budget_at_the_thresholds(batch, keys):
    """bfv.decrypt's budget is 72 - bit_count(noise) - 1 with the noise computed here; it is 1 at a centred remainder of
    2^70 - 1 and 0 at 2^70, on both sides of q / 2; the plaintexts equal the restated rounding"""
    want = {"2^70-1": 1, "2^70": 0, "q-2^70": 0, "q-2^70+1": 1, "(q-1)/2": 0, "(q+1)/2": 0}
    for ct, cls in zip(batch.dec, batch.dec_classes):
        (name,) = [c.split("=", 1)[1] for c in cls]
        for sk in (keys.sk, keys.net_sk):  # c1 = 0: the key does not matter
            plain, budget = bfv.decrypt(ct, sk)
            p, exhausted, b = E.decrypt_expect(ct)
            assert budget == b == want[name], name
            assert exhausted == (budget <= 0)
            assert np.array_equal(plain, p), name


def test_pipe_chunk_mirror_covers_every_branch():
    """the n values the host-pipeline tests run take every branch of engine.cpp's pipe_chunk at the default 256-op chunk"""
    seen = set()
    for n in E.PIPE_NS:
        sched = E.pipe_schedule(n, 256, seen)
        assert sum(sched) == n and all(0 < c <= 256 for c in sched)
    assert seen == set(E.PIPE_BRANCHES), sorted(set(E.PIPE_BRANCHES) - seen)
    assert E.pipe_schedule(150, 256) == [96, 54]  # a fused chunk, then a split one
    assert E.pipe_schedule(700, 256) == [96, 256, 252, 96]
