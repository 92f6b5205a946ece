"""Operands crafted to land exactly on the per-coefficient decisions of the multiply, key-switch and decrypt kernels.

Uniform residues almost never hit these decisions (2^-32 to 2^-37 per coefficient), so a kernel that is off by one at one of
them passes a suite of uniform inputs.  This module restates, in Python big integers, the variables the kernels branch on,
line for line with kernels.cu, and solves for residues that put each variable on its boundary:

  ext_vars      ext_shared (k_ext_conv_d): y0, y0 >= q, ymt, rm, neg = rm >= 2^31, the carry (ymt != 0), m, base
  floor_vars    floor_sk_coeff_d (k_floor_sk_d / k_tensor_floor_d): t0, t1, y0' of t D mod q, u2, y0' mod s_i
  ks_vars       the key switch's rounded division by P (k_ks_tail_ksd / k_relin_finish): U mod P, last
  decrypt_vars  k_decrypt_round: the remainder of t X mod q, up, nh, the exhausted flag, the plaintext

edge_batch() returns the crafted operands together with the classes each one covers.  No GPU is needed here.
"""
from __future__ import annotations

import functools
import importlib.util
import os
from dataclasses import dataclass, field
from typing import Dict, List, Set

import numpy as np

from helpers import N, ROOT, random_ct
from oracle import bfv

M32 = (1 << 32) - 1
MTILDE = 1 << 32
M64 = (1 << 64) - 1


@functools.lru_cache(None)
def _check_dual_base():
    spec = importlib.util.spec_from_file_location("check_dual_base", os.path.join(ROOT, "scripts", "check_dual_base.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@dataclass(frozen=True)
class Consts:
    q0: int
    q1: int
    P: int
    q: int
    t: int
    ext_in: tuple  # m~ (q / q_l)^-1 mod q_l: what ext_shared multiplies x_l by
    inv_punct_q: tuple  # (q / q_l)^-1 mod q_l
    neg_inv_q: int  # -q^-1 mod m~
    q_w: tuple  # the three 32-bit words of q
    half_P: int
    dual: tuple  # the six dual primes s_0 .. s_5


@functools.lru_cache(None)
def consts() -> Consts:
    c = bfv.constants()
    q0, q1, P = c["moduli"][:3]
    q = q0 * q1
    ext_in = tuple(c["mtilde_mod_q"][l] * c["inv_punct_q"][l] % ql for l, ql in enumerate((q0, q1)))
    return Consts(q0, q1, P, q, bfv.T, ext_in, tuple(c["inv_punct_q"]), c["neg_inv_q_mod_mtilde"],
                  (q & M32, (q >> 32) & M32, q >> 64), c["half_P"], tuple(_check_dual_base().dual_primes()))


# ---------------------------------------------------------------- restated decision variables
@functools.lru_cache(None)
def ext_vars(x0: int, x1: int) -> dict:
    """ext_shared(x0, x1): Z = base + m 2^61 - (q if neg) is the extended operand a' = (y0 + rm q) / m~, rm centred."""
    k = consts()
    t0 = x0 * k.ext_in[0] % k.q0
    t1 = x1 * k.ext_in[1] % k.q1
    y0 = t0 * k.q1 + t1 * k.q0  # punctured_sum
    ymt = y0 & M32
    rm = ymt * k.neg_inv_q & M32
    neg = rm >= 0x80000000
    carry = 1 if ymt != 0 else 0
    A = ((y0 >> 32) & M64) + ((rm * k.q_w[0]) >> 32) + carry
    Bv, Cv = rm * k.q_w[1], rm * k.q_w[2]
    sAB = (A + Bv) & M64
    wrap = sAB < A  # the "+ 8u" term: never set (test_edge_inputs bounds it)
    m = (sAB >> 61) + (8 if wrap else 0) + (Cv >> 29)
    base = (sAB & ((1 << 61) - 1)) + ((Cv & ((1 << 29) - 1)) << 32)
    Z = base + (m << 61) - (k.q if neg else 0)
    return dict(y0=y0, over=y0 >= k.q, ymt=ymt, rm=rm, neg=neg, carry=carry, A=A, sAB_wrap=wrap, m=m, base=base, Z=Z)


@functools.lru_cache(None)
def floor_vars(tD: int) -> dict:
    """floor_sk_coeff_d for one coefficient of t D (an exact integer): t_l = t D (q / q_l)^-1 mod q_l, y0' = t0 q1 + t1 q0
    (t D mod q, plus q when the fast conversion overflows), u2 = y0' >> 58, y0' mod s_i (i < 4), f = (t D - y0') / q."""
    k = consts()
    t0 = tD * k.inv_punct_q[0] % k.q0
    t1 = tD * k.inv_punct_q[1] % k.q1
    y0p = t0 * k.q1 + t1 * k.q0
    assert (tD - y0p) % k.q == 0
    return dict(t0=t0, t1=t1, y0p=y0p, over=y0p >= k.q, u2=y0p >> 58, ymod=[y0p % s for s in k.dual[:4]], f=(tD - y0p) // k.q)


def ks_vars(U: int) -> dict:
    """the rounded division by P: last = (U mod P + P/2) mod P; out_l = c_l + (U - (last - P/2)) P^-1 mod q_l"""
    k = consts()
    umod = U % k.P
    return dict(umodP=umod, last=(umod + k.half_P) % k.P)


def decrypt_vars(X: int) -> dict:
    """k_decrypt_round for X = CRT(x0, x1) in [0, q): quo, rem = divmod(t X, q); up iff rem + (q-1)/2 >= q; nh = bits 64.. of
    the centred remainder; exhausted iff nh >> 6 (centred remainder >= 2^70); plaintext (quo + up) mod t."""
    k = consts()
    quo, rem = divmod(k.t * X, k.q)
    up = rem + (k.q - 1) // 2 >= k.q
    centred = k.q - rem if up else rem
    nh = centred >> 64
    return dict(rem=rem, up=up, centred=centred, nh=nh, exhausted=(nh >> 6) != 0, plain=(quo + up) % k.t)


def bit_count(v: int) -> int:
    return v.bit_length()


# ---------------------------------------------------------------- classes
RM_TARGETS = (0, 1, (1 << 31) - 1, 1 << 31, (1 << 31) + 1, (1 << 32) - 1)
EXT_CLASSES = [f"ext:rm={r:#x}:{'over' if o else 'under'}" for r in RM_TARGETS for o in (False, True)] + \
    ["ext:carry0_y0_nonzero", "ext:x=(q-1)/2", "ext:x=(q+1)/2"]
FLOOR_TARGETS = ("y0p=q-1", "y0p=q+1", "tD=0", "tD>0", "tD<0", "max|AB|", "u2=0", "u2=max") + \
    tuple(f"y0p%s{i}={e}:{o}" for i in range(4) for e in ("0", "s-1") for o in ("under", "over"))
FLOOR_CLASSES = [f"floor:{c}:{w}" for c in FLOOR_TARGETS for w in ("nowrap", "wrap")]
KS_CLASSES = [f"ks:U%P={n}:k{k}" for n in ("(P-1)/2", "(P+1)/2", "0", "P-1") for k in (0, 1)] + ["ks:digits=q-1"]
DEC_CLASSES = [f"dec:rem={n}" for n in ("2^70-1", "2^70", "q-2^70", "q-2^70+1", "(q-1)/2", "(q+1)/2")]


def ext_classes(x0: int, x1: int) -> Set[str]:
    k = consts()
    v = ext_vars(x0, x1)
    out = set()
    if v["rm"] in RM_TARGETS:
        out.add(f"ext:rm={v['rm']:#x}:{'over' if v['over'] else 'under'}")
    if v["ymt"] == 0 and v["y0"] != 0:
        out.add("ext:carry0_y0_nonzero")
    x = _crt(x0, x1)
    if x == (k.q - 1) // 2:
        out.add("ext:x=(q-1)/2")
    if x == (k.q + 1) // 2:
        out.add("ext:x=(q+1)/2")
    return out


@functools.lru_cache(None)
def floor_classes(tD: int, A: int, B: int, wrap: bool) -> frozenset:
    k = consts()
    v = floor_vars(tD)
    names = set()
    if v["y0p"] == k.q - 1:
        names.add("y0p=q-1")
    if v["y0p"] == k.q + 1:
        names.add("y0p=q+1")
    names.add("tD=0" if tD == 0 else "tD>0" if tD > 0 else "tD<0")
    if abs(A * B) >= ((k.q - 1) // 2) ** 2:
        names.add("max|AB|")
    if v["u2"] == 0:
        names.add("u2=0")
    if v["u2"] == (2 * k.q - k.q0 - k.q1) >> 58:  # y0' <= (q0 - 1) q1 + (q1 - 1) q0
        names.add("u2=max")
    for i, s in enumerate(k.dual[:4]):
        for e, r in (("0", 0), ("s-1", s - 1)):
            if v["ymod"][i] == r:
                names.add(f"y0p%s{i}={e}:{'over' if v['over'] else 'under'}")
    w = "wrap" if wrap else "nowrap"
    return frozenset(f"floor:{c}:{w}" for c in names)


def _crt(x0: int, x1: int) -> int:
    k = consts()
    return (x0 * k.inv_punct_q[0] % k.q0 * k.q1 + x1 * k.inv_punct_q[1] % k.q1 * k.q0) % k.q


def _put(ct: np.ndarray, poly: int, idx, xs) -> None:
    """ct[poly][l][idx] = xs mod q_l (xs: python ints in [0, q))"""
    k = consts()
    xs = list(xs)
    ct[poly, 0, idx] = np.array([x % k.q0 for x in xs], dtype=np.uint64)
    ct[poly, 1, idx] = np.array([x % k.q1 for x in xs], dtype=np.uint64)


def _ints(ct: np.ndarray, poly: int) -> List[int]:
    return [_crt(int(a), int(b)) for a, b in zip(ct[poly, 0], ct[poly, 1])]


# ---------------------------------------------------------------- extension crafting
def craft_ext(rng: np.random.Generator, per_class: int = 8) -> Dict[str, List[int]]:
    """x in [0, q) per class: y0 = -R q (mod 2^32) gives rm = R; x = y0 m~^-1 mod q, kept when the restatement confirms
    (the conversion decides whether y0 is the residue or the residue + q)."""
    k = consts()
    minv = pow(MTILDE, -1, k.q)
    pool: Dict[str, List[int]] = {c: [] for c in EXT_CLASSES}
    for R in RM_TARGETS:
        T = (-R * k.q) % MTILDE
        for over in (False, True):
            name = f"ext:rm={R:#x}:{'over' if over else 'under'}"
            for _ in range(2000):
                lo = k.q if over else 0
                y = T + MTILDE * int(rng.integers((lo + MTILDE - 1 - T) // MTILDE, (lo + k.q - T) // MTILDE))
                x = y % k.q * minv % k.q
                got = ext_classes(x % k.q0, x % k.q1)
                if name in got:
                    pool[name].append(x)
                    if "ext:carry0_y0_nonzero" in got:
                        pool["ext:carry0_y0_nonzero"].append(x)
                    if len(pool[name]) == per_class:
                        break
    pool["ext:x=(q-1)/2"] = [(k.q - 1) // 2]
    pool["ext:x=(q+1)/2"] = [(k.q + 1) // 2]
    return pool


# ---------------------------------------------------------------- floor crafting (monomial operands)
FLOOR_SHIFTS = (0, 1, N // 2, N - 1)


def _floor_residues(rng: np.random.Generator) -> List[tuple]:
    """(target name, R = t D mod q) pairs whose y0' the restatement confirms; R = None: b's coefficient is 0 (t D = 0) or one of
    the lifts (q -+ 1)/2 (largest |B|)"""
    k = consts()
    out = [("y0p=q-1", k.q - 1), ("y0p=q+1", 1), ("tD=0", None), ("max|AB|", None)]
    while True:  # y0' < 2^58: a small t D mod q that the conversion does not overflow
        R = int(rng.integers(1, 1 << 57))
        if floor_vars(R)["u2"] == 0:
            out.append(("u2=0", R))
            break
    out.append(("u2=max", k.q - k.q0 - k.q1))  # t_l = q_l - 1: y0' = (q0 - 1) q1 + (q1 - 1) q0 = R + q, its largest value
    for i, s in enumerate(k.dual[:4]):
        for e, r in (("0", 0), ("s-1", s - 1)):
            for over in (False, True):
                for tries in range(1000):
                    R = int(rng.integers(0, k.q // s - 1)) * s + (r - (k.q if over else 0)) % s  # y0' = R (+ q) = r mod s
                    v = floor_vars(R)
                    if v["ymod"][i] == r and v["over"] == over:
                        out.append((f"y0p%s{i}={e}:{'over' if over else 'under'}", R))
                        break
                else:
                    raise AssertionError(f"no t D mod q with y0' = {e} mod s_{i}")
    return out


def craft_floor_op(targets: List[tuple], j: int, xa: int, phase: int):
    """a = (xa X^j, 0), b chosen coefficient by coefficient: with a'_1 = 0 the tensor is D_0 = A X^j b'_0, D_1 = A X^j b'_1,
    so t D_d[i] = +-t A B_d[i - j] (sign - where i - j wraps) and each b coefficient targets its own t D mod q."""
    k = consts()
    a = np.zeros((2, 2, N), dtype=np.uint64)
    _put(a, 0, [j], [xa])
    inv = {s: pow(s * k.t * xa % k.q, -1, k.q) for s in (1, -1)}
    b = np.zeros((2, 2, N), dtype=np.uint64)
    for p in range(2):
        xs = []
        for kk in range(N):
            name, R = targets[(kk + phase + 7 * p) % len(targets)]
            sign = -1 if kk + j >= N else 1
            if name == "tD=0":
                xs.append(0)
            elif R is None:
                xs.append((k.q - 1) // 2 + (kk & 1))
            else:
                xs.append(R * inv[sign] % k.q)
        _put(b, p, slice(None), xs)
    return a, b


def floor_coverage(a: np.ndarray, b: np.ndarray) -> Set[str]:
    """classes hit by the product of a monomial a = (x X^j, 0) with any b (recomputed from the restatements)"""
    nz = np.nonzero(a[0, 0] | a[0, 1])[0]
    assert len(nz) == 1 and not a[1].any()
    j = int(nz[0])
    A = ext_vars(int(a[0, 0, j]), int(a[0, 1, j]))["Z"]
    t = consts().t
    out = set()
    for p in range(2):
        for kk in range(N):
            B = ext_vars(int(b[p, 0, kk]), int(b[p, 1, kk]))["Z"]
            wrap = kk + j >= N
            out |= floor_classes(t * A * B * (-1 if wrap else 1), A, B, wrap)
    return out


def floor_product(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """the size-3 product of a monomial a with b from the restatements alone: limb l of c3[d][i] = f mod q_l"""
    k = consts()
    j = int(np.nonzero(a[0, 0] | a[0, 1])[0][0])
    A = ext_vars(int(a[0, 0, j]), int(a[0, 1, j]))["Z"]
    out = np.zeros((3, 2, N), dtype=np.uint64)
    for p in range(2):
        for kk in range(N):
            B = ext_vars(int(b[p, 0, kk]), int(b[p, 1, kk]))["Z"]
            i, sign = (kk + j) % N, -1 if kk + j >= N else 1
            f = floor_vars(k.t * A * B * sign)["f"]
            out[p, 0, i], out[p, 1, i] = f % k.q0, f % k.q1
    return out


# ---------------------------------------------------------------- key-switch crafting
def rk_integers(rk: np.ndarray) -> Dict[tuple, List[int]]:
    """RK[j, k]: the coefficient-form key lifted to integers (== rk mod q0, q1, P; 0 <= RK < q0 q1 P)"""
    k = consts()
    ms = (k.q0, k.q1, k.P)
    Q = k.q0 * k.q1 * k.P
    w = [pow(Q // m, -1, m) for m in ms]
    out = {}
    for j in range(2):
        for kk in range(2):
            coef = [bfv.ntt_inv(rk[j, kk, mi].copy(), mi) for mi in range(3)]
            out[j, kk] = [sum(int(coef[mi][i]) * w[mi] % m * (Q // m) for mi, m in enumerate(ms)) % Q for i in range(N)]
    return out


def ks_U(c3: np.ndarray, RK, kk: int, i: int) -> int:
    """U_k[i] = sum_j d_j * RK_jk at coefficient i for monomial digits (d_j = [c2]_{q_j}, both at the same power or zero)"""
    U = 0
    for jd in range(2):
        nz = np.nonzero(c3[2, jd])[0]
        assert len(nz) <= 1
        if len(nz):
            p = int(nz[0])
            src = (i - p) % N
            U += int(c3[2, jd, p]) * RK[jd, kk][src] * (-1 if i < p else 1)
    return U


def _uniform_c3(rng: np.random.Generator) -> np.ndarray:
    return random_ct(rng, 2).reshape(4, 2, N)[:3].copy()


KS_TARGETS = (("(P-1)/2", lambda P: (P - 1) // 2), ("(P+1)/2", lambda P: (P + 1) // 2), ("0", lambda P: 0), ("P-1", lambda P: P - 1))


def craft_ks(rng: np.random.Generator, RK) -> tuple:
    """size-3 ciphertexts (c0, c1 uniform) whose c2 has digit 0 = c X^j and digit 1 = e X^j (e = 0 unless the target is
    U mod P = 0, which a single non-zero digit cannot give): c solved mod P so that U_k mod P hits the target at a random
    coefficient, kept when c < q0.  Plus digits q_j - 1 everywhere."""
    k = consts()
    cts, cls = [], []
    for name, tf in KS_TARGETS:
        T = tf(k.P)
        for kk in range(2):
            for j in (0, N // 2):
                for _ in range(200):
                    i = int(rng.integers(0, N))
                    e = 0 if T else int(rng.integers(1, k.q1))
                    sign = -1 if i < j else 1
                    r0 = sign * RK[0, kk][(i - j) % N] % k.P
                    r1 = sign * RK[1, kk][(i - j) % N] % k.P
                    c = (T - e * r1) * pow(r0, -1, k.P) % k.P
                    if 0 < c < k.q0:
                        break
                else:
                    raise AssertionError("no key-switch digit found")
                c3 = _uniform_c3(rng)
                c3[2] = 0
                c3[2, 0, j], c3[2, 1, j] = c, e
                assert ks_vars(ks_U(c3, RK, kk, i))["umodP"] == T
                cts.append(c3)
                cls.append({f"ks:U%P={name}:k{kk}"})
    c3 = _uniform_c3(rng)
    c3[2, 0], c3[2, 1] = k.q0 - 1, k.q1 - 1
    cts.append(c3)
    cls.append({"ks:digits=q-1"})
    return np.stack(cts), cls


# ---------------------------------------------------------------- decrypt crafting
DEC_TARGETS = (("2^70-1", lambda q: (1 << 70) - 1), ("2^70", lambda q: 1 << 70), ("q-2^70", lambda q: q - (1 << 70)),
               ("q-2^70+1", lambda q: q - (1 << 70) + 1), ("(q-1)/2", lambda q: (q - 1) // 2), ("(q+1)/2", lambda q: (q + 1) // 2))


def craft_decrypt(rng: np.random.Generator) -> tuple:
    """c1 = 0 (the result does not depend on the key), c0 = CRT(X): every coefficient is a plaintext with little noise
    (X = round(q m / t)) except a few at which t X mod q is the target remainder.  One target per ciphertext, so its exhausted
    flag is decided by that target alone."""
    k = consts()
    tinv = pow(k.t, -1, k.q)
    cts, cls = [], []
    for name, tf in DEC_TARGETS:
        R = tf(k.q)
        ms = rng.integers(0, k.t, size=N)
        xs = [(int(m) * k.q + k.t // 2) // k.t for m in ms]
        for i in rng.choice(N, size=16, replace=False):
            xs[int(i)] = (R + int(rng.integers(0, k.t)) * k.q) * tinv % k.q  # t X = R (mod q), any quotient
        ct = np.zeros((2, 2, N), dtype=np.uint64)
        _put(ct, 0, slice(None), xs)
        cts.append(ct)
        cls.append({f"dec:rem={name}"})
    return np.stack(cts), cls


def decrypt_expect(ct: np.ndarray) -> tuple:
    """(plaintext [N], exhausted, budget) of a c1 = 0 ciphertext from decrypt_vars alone"""
    assert not ct[1].any()
    vs = [decrypt_vars(x) for x in _ints(ct, 0)]
    noise = max(v["centred"] for v in vs)
    return np.array([v["plain"] for v in vs], dtype=np.uint64), any(v["exhausted"] for v in vs), 72 - bit_count(noise) - 1


# ---------------------------------------------------------------- the batch
@dataclass
class EdgeBatch:
    a: np.ndarray  # [n][2][2][N] multiply operands
    b: np.ndarray
    kind: List[str]  # per op: "ext", "floor", "mixed" (uniform with crafted coefficients) or "uniform"
    classes: List[Set[str]]  # per op: the classes its coefficients cover
    c3: np.ndarray = field(default=None)  # [m][3][2][N] size-3 key-switch operands
    c3_classes: List[Set[str]] = field(default=None)
    dec: np.ndarray = field(default=None)  # [6][2][2][N] decrypt operands
    dec_classes: List[Set[str]] = field(default=None)


@functools.lru_cache(None)
def _rk_integers_cached(key: bytes):
    return rk_integers(np.frombuffer(key, dtype=np.uint64).reshape(2, 2, 3, N))


def edge_batch(rk: np.ndarray = None, n: int = 256, seed: int = 2024) -> EdgeBatch:
    """n >= 256 multiply operand pairs: 96 built from the extension pool alone (every coefficient on an ext_shared boundary),
    64 floor monomial pairs (4 shifts x 2 monomial values x 8 phases of the target cycle), 56 uniform pairs with one crafted
    coefficient in eight, the rest uniform.  With rk: the crafted size-3 key-switch ciphertexts for that key.  Always: the six
    crafted decrypt ciphertexts."""
    assert n >= 256
    k = consts()
    rng = np.random.default_rng(seed)
    pool = craft_ext(rng)
    flat = [(x, c) for c, xs in pool.items() for x in xs]
    flat = [(x, *ext_classes(x % k.q0, x % k.q1)) for x, _ in flat]
    vals = np.array([x for x, *_ in flat], dtype=object)
    targets = _floor_residues(rng)
    a, b = random_ct(rng, n), random_ct(rng, n)
    kind, classes = [], []
    for i in range(n):
        if i < 96:
            used = set()
            for ct in (a[i], b[i]):
                for p in range(2):
                    pick = rng.integers(0, len(vals), size=N)
                    _put(ct, p, slice(None), vals[pick])
                    used.update(pick.tolist())
            kind.append("ext")
            classes.append(set().union(*(flat[u][1:] for u in used)))
        elif i < 160:
            r = i - 96
            j = FLOOR_SHIFTS[r % 4]
            # the largest |A| in odd groups of four; otherwise any A invertible mod q (both residues non-zero)
            xa = (k.q - 1) // 2 if (r // 4) % 2 else _crt(int(rng.integers(1, k.q0)), int(rng.integers(1, k.q1)))
            a[i], b[i] = craft_floor_op(targets, j, xa, r // 8)
            kind.append("floor")
            classes.append(None)  # filled below from the restatements
        elif i < 216:
            used = set()
            for ct in (a[i], b[i]):
                for p in range(2):
                    pick = rng.integers(0, len(vals), size=N // 8)
                    _put(ct, p, rng.choice(N, size=N // 8, replace=False), vals[pick])
                    used.update(pick.tolist())
            kind.append("mixed")
            classes.append(set().union(*(flat[u][1:] for u in used)))
        else:
            kind.append("uniform")
            classes.append(set())
    for i in range(n):
        if kind[i] == "floor":
            classes[i] = floor_coverage(a[i], b[i])
    batch = EdgeBatch(a, b, kind, classes)
    if rk is not None:
        RK = _rk_integers_cached(np.ascontiguousarray(rk, dtype=np.uint64).tobytes())
        batch.c3, batch.c3_classes = craft_ks(rng, RK)
    batch.dec, batch.dec_classes = craft_decrypt(rng)
    return batch


def _pairs(*cts) -> np.ndarray:
    """the distinct residue pairs (x0, x1) of the coefficients of ciphertexts [2][2][N]"""
    p = np.concatenate([np.stack([c[:, 0].ravel(), c[:, 1].ravel()], axis=1) for c in cts])
    return np.unique(p, axis=0)


# ---------------------------------------------------------------- the host pipelines' chunk schedule
FUSED_TAIL_MIN_OPS = 96  # engine.cpp kFusedTailMinOps: chunks of at least this many ops run the fused tails
PIPE_BRANCHES = ("small", "first", "last>2edge", "last", "second-last", "full")
PIPE_NS = (1, 95, 96, 97, 150, 192, 193, 289, 353, 700)  # every branch at the default 256-op chunk


def pipe_chunk(off: int, n: int, chunk: int, seen: set = None) -> int:
    """engine.cpp pipe_chunk, branch for branch; `seen` collects the branches taken"""
    rem, edge = n - off, FUSED_TAIL_MIN_OPS
    take = (lambda b, v: (seen.add(b), v)[1]) if seen is not None else (lambda b, v: v)
    if chunk <= edge or rem <= edge:
        return take("small", rem if rem < chunk else chunk)
    if off == 0:
        return take("first", edge)
    if rem <= chunk:
        return take("last>2edge", rem - edge) if rem > 2 * edge else take("last", rem)
    if rem <= chunk + edge:
        return take("second-last", rem - edge)
    return take("full", chunk)


def pipe_schedule(n: int, chunk: int, seen: set = None) -> List[int]:
    out, off = [], 0
    while off < n:
        out.append(pipe_chunk(off, n, chunk, seen))
        off += out[-1]
    return out
