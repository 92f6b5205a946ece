"""The algebra behind the GPU's dual auxiliary base (DESIGN.md section 4), checked against the oracle (which follows SEAL)
before any kernel was written -- pure CPU:

  * bfv_multiply: the extended operands a' are integers, D = a' * b' (negacyclic, over Z) has |t D| < 2^166, so carrying it
    on six NTT primes below 2^30 (product 2^180), recovering t_l = t D (q/q_l)^-1 mod q_l by CRT with rounding, forming
    y0 = t_0 q_1 + t_1 q_0 and lifting f = (t D - y0) / q from four of the primes by rounding gives SEAL's size-3 result bit
    for bit;
  * key switch (what the library runs for chunks of 96 ops and more): U_k = sum_j d_j * RK_jk over Z with the key lifted to integers, |U_k| < 2^161,
    carried on the same six primes; U_k mod (q0, q1, P) by the same CRT gives SEAL's relinearised ciphertext bit for bit.

usage: python scripts/check_dual_base.py [pairs]      (tests/test_integer_domain.py runs one pair)"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import bfv  # noqa: E402

N = 4096
T = 4096


def is_prime(n: int) -> bool:
    if n < 2:
        return False
    for p in (2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37):
        if n % p == 0:
            return n == p
    d, s = n - 1, 0
    while d % 2 == 0:
        d //= 2
        s += 1
    for a in (2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37):
        x = pow(a, d, n)
        if x in (1, n - 1):
            continue
        for _ in range(s - 1):
            x = x * x % n
            if x == n - 1:
                break
        else:
            return False
    return True


def dual_primes():
    """the six largest primes below 2^30 that are 1 mod 2N (params.h: kDualPrime)"""
    out, v = [], ((1 << 30) - 1) // (2 * N) * (2 * N) + 1
    while len(out) < 6:
        if is_prime(v):
            out.append(v)
        v -= 2 * N
    return out


def _root(q: int) -> int:
    cof, g = (q - 1) // (2 * N), 2
    while True:
        c = pow(g, cof, q)
        if pow(c, N, q) == q - 1:
            return c
        g += 1


def negacyclic_mul(a: np.ndarray, b: np.ndarray, q: int) -> np.ndarray:
    """a * b mod (x^N + 1, q) for q < 2^30 (int64 numpy, recursive radix-2)"""
    psi = _root(q)
    w = psi * psi % q
    pw = np.array([pow(psi, i, q) for i in range(N)], dtype=np.int64)
    ipw = np.array([pow(psi, -i, q) for i in range(N)], dtype=np.int64)

    def ntt(x, root):
        n = len(x)
        if n == 1:
            return x
        e, o = ntt(x[0::2], root * root % q), ntt(x[1::2], root * root % q)
        tw = np.array([pow(root, i, q) for i in range(n // 2)], dtype=np.int64)
        t = o * tw % q
        return np.concatenate([(e + t) % q, (e - t) % q])

    c = ntt(ntt(a * pw % q, w) * ntt(b * pw % q, w) % q, pow(w, -1, q))
    return c * pow(N, -1, q) % q * ipw % q


def crt_round(res, primes):
    """exact signed integer from residues res[i] mod primes[i] when |X| << prod / 2: y_i, v = round(sum y_i / s_i) from 16-bit
    estimates by shifts (every prime is within 2^-12 of 2^30), as the kernels do"""
    S = 1
    for p in primes:
        S *= p
    y = [res[i] * pow(S // primes[i], -1, primes[i]) % primes[i] for i in range(len(primes))]
    v = (sum(yi >> 14 for yi in y) + (1 << 15)) >> 16
    return sum(y[i] * (S // primes[i]) for i in range(len(primes))) - v * S


def check_multiply(a: np.ndarray, b: np.ndarray) -> int:
    q0, q1, P, b0, b1, msk = bfv.moduli()
    q = q0 * q1
    primes = dual_primes()
    ext = bfv.behz_extend(a, b)  # [4][5][N]: a' mod (q0, q1, b0, b1, m_sk)
    B3 = b0 * b1 * msk
    ints = []
    for p in range(4):  # the integers a' themselves (|a'| <= q/2 (1 + 2^-30)), from the oracle's Bsk residues
        r = [ext[p, 2 + i].astype(object) for i in range(3)]
        X = sum(r[i] * pow(B3 // m, -1, m) % m * (B3 // m) for i, m in enumerate((b0, b1, msk))) % B3
        X = np.where(X > B3 // 2, X - B3, X)
        assert max(abs(int(x)) for x in X) <= (q // 2) * (1 + 2 ** -29)
        ints.append(X)
    want = bfv.multiply(a, b)
    bad = 0
    for d in range(3):
        res = []
        for s in primes:
            A0, A1, B0, B1 = (np.array([int(x) % s for x in ints[k]], dtype=np.int64) for k in range(4))
            D = negacyclic_mul(A0, B0, s) if d == 0 else negacyclic_mul(A1, B1, s) if d == 2 else \
                (negacyclic_mul(A0, B1, s) + negacyclic_mul(A1, B0, s)) % s
            res.append((D * T % s).astype(object))
        X = crt_round(res, primes)
        assert max(abs(int(x)) for x in X) < 2 ** 166
        t = [X * pow(q // ql, -1, ql) % ql for ql in (q0, q1)]
        y0 = t[0] * q1 + t[1] * q0
        f = crt_round([(res[i] - y0) % primes[i] * pow(q, -1, primes[i]) % primes[i] for i in range(4)], primes[:4])
        assert max(abs(int(x)) for x in f) < 2 ** 97
        for l, ql in enumerate((q0, q1)):
            bad += int(((f % ql) != want[d, l].astype(object)).sum())
    return bad


def check_key_switch(c3: np.ndarray, rk: np.ndarray) -> int:
    q0, q1, P = bfv.moduli()[:3]
    ms, Q = (q0, q1, P), q0 * q1 * P
    primes = dual_primes()
    want = bfv.relinearize(c3, rk)
    RK = {}
    for j in range(2):
        for k in range(2):
            acc = np.zeros(N, dtype=object)
            for mi, m in enumerate(ms):
                coef = bfv.ntt_inv(rk[j, k, mi].copy(), mi).astype(object)
                acc = acc + coef * pow(Q // m, -1, m) % m * (Q // m)
            RK[j, k] = acc  # == rk mod every m, 0 <= RK < 3 Q
    bad = 0
    for k in range(2):
        res = []
        for s in primes:
            u = np.zeros(N, dtype=np.int64)
            for j in range(2):
                d = np.array([int(x) % s for x in c3[2, j]], dtype=np.int64)
                K = np.array([int(x) % s for x in RK[j, k]], dtype=np.int64)
                u = (u + negacyclic_mul(d, K, s)) % s
            res.append(u.astype(object))
        U = crt_round(res, primes)
        assert max(abs(int(x)) for x in U) < 2 ** 161
        half = P >> 1
        last = (U % P + half) % P
        for l, ql in enumerate((q0, q1)):
            tl = (last % ql - half % ql) % ql
            out = (c3[k, l].astype(object) + (U % ql - tl) * pow(P, -1, ql)) % ql
            bad += int((out != want[k, l].astype(object)).sum())
    return bad


def main():
    from helpers import KeySet, encrypt_value, random_ct

    pairs = int(sys.argv[1]) if len(sys.argv) > 1 else 2
    keys = KeySet.load()
    primes = dual_primes()
    print("dual primes:", [hex(p) for p in primes], "product 2^%.2f" % sum(np.log2(primes)))
    rng = np.random.default_rng(5)
    for i in range(pairs):
        a, b = (random_ct(rng, 2)) if i else (encrypt_value(keys, "i64", 5, 1), encrypt_value(keys, "i64", -9, 2))
        print("pair", i, "multiply mismatches:", check_multiply(a, b))
        c3 = np.concatenate([a, b[:1]])
        print("pair", i, "key switch mismatches:", check_key_switch(c3, keys.rk))


if __name__ == "__main__":
    main()
