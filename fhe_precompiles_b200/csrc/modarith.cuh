// 64-bit modular arithmetic on the sm_100a integer pipes.
// Replaces SEAL util/uintarithsmallmod.h (barrett_reduce_64/128, MultiplyUIntModOperand)
// on the reference's hot path (FheApp::run, /root/reference/src/fhe.rs:138-152).
//
// B200 has two integer issue paths per SM sub-partition, each 16 lanes wide: the FMA pipe (IMAD,
// IMAD.WIDE) and the ALU pipe (IADD3, LOP3, SEL, ISETP, SHF).  Everything here is written on 32-bit
// halves so that the multiply-accumulate chains carry on the FMA pipe (IMAD.WIDE accumulates 64 bits
// for free) and only the unavoidable adds / selects land on the ALU pipe; the first version (plain
// __umul64hi + 64-bit adds) was ALU-bound at 2 ALU : 1 FMA instructions (profiles/r1a).
//
// Two prime classes, selected at compile time by Mod<MI>::kSmall:
//  * 36/37-bit data and key-switch primes (q0, q1, P) = 2^b - c with c < 2^18: 27 bits of headroom in a
//    word, so butterflies never conditionally subtract, the Shoup quotient drops its lowest partial
//    product, and reduction is a pseudo-Mersenne fold.
//  * 61-bit BEHZ primes (b0, b1, m_sk) = 2^61 - c: Harvey-style lazy ranges with a conditional
//    subtraction every other forward stage ([0,8q) fits a word).
#pragma once
#include "params.h"

namespace fheb {

constexpr int mod_bits(u64 q) {
    int b = 0;
    while (q) {
        b++;
        q >>= 1;
    }
    return b;
}

template <int MI>
struct Mod {
    static constexpr bool kDual = false;
    static constexpr int kIndex = MI;
    static constexpr u64 q = kModulus[MI];
    static constexpr u64 two_q = 2 * kModulus[MI];
    static constexpr u64 four_q = 4 * kModulus[MI];
    static constexpr u64 r1 = barrett_ratio(kModulus[MI]).hi;  // floor(2^64/q)
    static constexpr u64 r0 = barrett_ratio(kModulus[MI]).lo;
    static constexpr bool kSmall = kModulus[MI] < (1ull << 40);
    static constexpr int kBits = mod_bits(kModulus[MI]);           // q < 2^kBits
    static constexpr u64 kC = (1ull << kBits) - kModulus[MI];      // q = 2^kBits - kC, kC < 2^19
    static constexpr u64 kMask = (1ull << kBits) - 1;
    static constexpr u64 neg_q = 0 - kModulus[MI];                 // -q mod 2^64
};

// 32-bit building blocks as PTX so that ptxas sees exactly the partial products we want
__device__ __forceinline__ void unpack64(u64 x, u32 &lo, u32 &hi) { asm("mov.b64 {%0,%1}, %2;" : "=r"(lo), "=r"(hi) : "l"(x)); }
__device__ __forceinline__ u64 pack64(u32 lo, u32 hi) {
    u64 r;
    asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "r"(lo), "r"(hi));
    return r;
}
__device__ __forceinline__ u64 mul_wide(u32 a, u32 b) {
    u64 r;
    asm("mul.wide.u32 %0, %1, %2;" : "=l"(r) : "r"(a), "r"(b));
    return r;
}
__device__ __forceinline__ u64 mad_wide(u32 a, u32 b, u64 c) {
    u64 r;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(r) : "r"(a), "r"(b), "l"(c));
    return r;
}
__device__ __forceinline__ u32 mad_lo(u32 a, u32 b, u32 c) {
    u32 r;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

__device__ __forceinline__ u64 mulhi64(u64 a, u64 b) { return __umul64hi(a, b); }

// (hi:lo) += a * b
__device__ __forceinline__ void mac128(u64 &lo, u64 &hi, u64 a, u64 b) {
    asm("mad.lo.cc.u64 %0, %2, %3, %0;\n\t"
        "madc.hi.u64 %1, %2, %3, %1;"
        : "+l"(lo), "+l"(hi)
        : "l"(a), "l"(b));
}

template <class M>
__device__ __forceinline__ u64 csub(u64 x, u64 m) {
    return x >= m ? x - m : x;
}

// acc + x*w - H*q (mod 2^64) with H ~ floor(x*ws/2^64): Shoup multiplication by the precomputed pair
// (w, ws = floor(w*2^64/q)) fused with an accumulate.  q = 2^B - c, so -H*q = H*c - (H << B).
//   exact quotient : adds a value in [0, 2q) for any 64-bit x
//   approximate 1  : drops the x_lo*ws_lo partial product and one carry (H low by <= 2): adds [0, 4q)
//   approximate 2  : x < 2^44 only; also estimates the x_hi*ws_lo term from 16 bits (H low by <= 3): adds [0, 5q)
// FMA pipe per call (IMAD.WIDE 4 cycles, IMAD 2): exact 6+4 (32), approximate 1: 5+4 (28), approximate 2: 4+5 (26).
// kApprox: 0 exact, 1 approximate for any 64-bit x ([0,4q)), 2 approximate for x < 2^44 ([0,5q), one wide multiply fewer)
template <class M, int kApprox>
__device__ __forceinline__ u64 shoup_acc(u64 acc, u64 x, u64 w, u64 ws) {
    constexpr u32 c = (u32)M::kC;
    u32 xl, xh, wl, wh, sl, sh;
    unpack64(x, xl, xh);
    unpack64(w, wl, wh);
    unpack64(ws, sl, sh);
    u64 H;
    if (kApprox == 2) {
        // x < 2^44, so xh < 2^12 and floor(xh*sl / 2^32) is estimated from the top 16 bits of sl with one low
        // multiply (IMAD: half the FMA-pipe cost of IMAD.WIDE); the estimate is low by at most 1
        u32 vl, vh;
        const u32 uh = (xh * (sl >> 16)) >> 16;
        unpack64(mul_wide(xl, sh), vl, vh);
        H = mad_wide(xh, sh, pack64(uh, 0)) + vh;
    } else if (kApprox == 1) {
        u32 ul, uh, vl, vh;
        unpack64(mul_wide(xh, sl), ul, uh);
        unpack64(mul_wide(xl, sh), vl, vh);
        H = mad_wide(xh, sh, pack64(uh, 0)) + vh;
    } else {
        // the middle column as one three-input add with two carries (ALU pipe): a multiply-add whose addend has a zero
        // high word is split by ptxas into IMAD.WIDE + IADD3 + IMAD.X, and the IMAD.X occupies the multiplier pipe
        u32 tl, th, ul, uh, vl, vh;
        unpack64(mul_wide(xl, sl), tl, th);
        unpack64(mul_wide(xh, sl), ul, uh);
        unpack64(mul_wide(xl, sh), vl, vh);
        const u64 mc = (u64)ul + (u64)vl + (u64)th;
        H = mul_wide(xh, sh) + (u64)uh + (u64)vh + (mc >> 32);
    }
    u32 hl, hh, al, ah;
    unpack64(H, hl, hh);
    u64 a = mad_wide(xl, wl, acc);
    a = mad_wide(hl, c, a);
    unpack64(a, al, ah);
    ah = mad_lo(xl, wh, ah);
    ah = mad_lo(xh, wl, ah);
    ah = mad_lo(hh, c, ah);
    ah -= hl << (M::kBits - 32);
    return pack64(al, ah);
}
// x*w mod q, lazy: [0, 2q) for any 64-bit x
template <class M>
__device__ __forceinline__ u64 shoup_lazy(u64 x, u64 w, u64 ws) {
    return shoup_acc<M, 0>(0, x, w, ws);
}
template <class M>
__device__ __forceinline__ u64 shoup(u64 x, u64 w, u64 ws) {
    return csub<M>(shoup_lazy<M>(x, w, ws), M::q);
}

// ---------------------------------------------------------------- dual limbs: two primes below 2^30 in one 64-bit word
// (params.h: kDualPrime).  32-bit Harvey arithmetic: values live in [0, 4s) < 2^32, a product by a precomputed pair
// (w, ws = floor(w 2^32 / s)) is one IMAD.HI + two IMAD and lands in [0, 2s) for ANY 32-bit operand.
template <int D>
struct ModDual {
    static constexpr bool kDual = true;
    static constexpr bool kSmall = false;
    static constexpr int kIndex = kNumMod + D;  // twiddle-table index
    static constexpr u32 s0 = kDualPrime[2 * D], s1 = kDualPrime[2 * D + 1];
};
__device__ __forceinline__ u32 shoup32(u32 x, u32 w, u32 ws, u32 s) { return x * w - __umulhi(x, ws) * s; }  // [0, 2s)
__device__ __forceinline__ u32 csub32(u32 x, u32 m) { return min(x, x - m); }                                // [0, 2m) -> [0, m)
// V < 2^61 -> V mod s in [0, 4s): q^ = floor(floor(V / 2^29) mu / 2^32), mu = floor(2^61 / s), is low by at most 3
__device__ __forceinline__ u32 barrett61(u64 V, u32 mu61, u32 s) { return (u32)V - __umulhi((u32)(V >> 29), mu61) * s; }
// one lane of the dyadic tensor: operands in [0, 4s) -> product(s) mod s in [0, 2s)
template <int NP>
__device__ __forceinline__ u32 dual_mulsum(const u32 (&x)[NP], const u32 (&y)[NP], u32 s, u32 mu61) {
    u64 P = 0;
#pragma unroll
    for (int k = 0; k < NP; k++) {
        const u32 a = csub32(csub32(x[k], 2 * s), s), b = csub32(csub32(y[k], 2 * s), s);  // canonical: a b < 2^60
        P = mad_wide(a, b, P);
    }
    return csub32(barrett61(P, mu61, s), 2 * s);
}
// forward butterfly on both lanes: inputs in [0, 4s), outputs in [0, 4s)
template <class M>
__device__ __forceinline__ void dual_fwd_bfly(u64 &X, u64 &Y, u64 w, u64 ws) {
    u32 x0, x1, y0, y1, w0, w1, q0, q1;
    unpack64(X, x0, x1);
    unpack64(Y, y0, y1);
    unpack64(w, w0, w1);
    unpack64(ws, q0, q1);
    x0 = csub32(x0, 2 * M::s0), x1 = csub32(x1, 2 * M::s1);
    const u32 t0 = shoup32(y0, w0, q0, M::s0), t1 = shoup32(y1, w1, q1, M::s1);
    const u32 z = kc.opaque_zero;  // a third addend: IADD3 on the ALU pipe instead of IMAD.IADD on the multiplier pipe
    X = pack64(x0 + t0 + z, x1 + t1 + z);
    Y = pack64(x0 + 2 * M::s0 - t0, x1 + 2 * M::s1 - t1);
}
// inverse butterfly: inputs in [0, 2s), outputs in [0, 2s)
template <class M>
__device__ __forceinline__ void dual_inv_bfly(u64 &X, u64 &Y, u64 w, u64 ws) {
    u32 x0, x1, y0, y1, w0, w1, q0, q1;
    unpack64(X, x0, x1);
    unpack64(Y, y0, y1);
    unpack64(w, w0, w1);
    unpack64(ws, q0, q1);
    const u32 d0 = x0 + 2 * M::s0 - y0, d1 = x1 + 2 * M::s1 - y1;
    const u32 z = kc.opaque_zero;
    X = pack64(csub32(x0 + y0 + z, 2 * M::s0), csub32(x1 + y1 + z, 2 * M::s1));
    Y = pack64(shoup32(d0, w0, q0, M::s0), shoup32(d1, w1, q1, M::s1));
}
// last inverse stage with the output scaling merged in: (X, Y) -> (sc (X + Y), scw (X - Y)), canonical if kCanon
template <class M, bool kCanon>
__device__ __forceinline__ void dual_inv_bfly_last(u64 &X, u64 &Y, u64 sc, u64 scs, u64 scw, u64 scws) {
    u32 x0, x1, y0, y1, a0, a1, b0, b1, c0, c1, e0, e1;
    unpack64(X, x0, x1);
    unpack64(Y, y0, y1);
    unpack64(sc, a0, a1);
    unpack64(scs, b0, b1);
    unpack64(scw, c0, c1);
    unpack64(scws, e0, e1);
    u32 s_0 = shoup32(x0 + y0, a0, b0, M::s0), s_1 = shoup32(x1 + y1, a1, b1, M::s1);
    u32 d_0 = shoup32(x0 + 2 * M::s0 - y0, c0, e0, M::s0), d_1 = shoup32(x1 + 2 * M::s1 - y1, c1, e1, M::s1);
    if (kCanon) s_0 = csub32(s_0, M::s0), s_1 = csub32(s_1, M::s1), d_0 = csub32(d_0, M::s0), d_1 = csub32(d_1, M::s1);
    X = pack64(s_0, s_1);
    Y = pack64(d_0, d_1);
}

// Exact sum of up to seven products x_k * w_k with x_k < 2^31 (a dual-lane residue in [0, 2s)) and constants w_k < q < 2^37,
// reduced ONCE: the low 30 bits of every w_k feed `lo` (each product < 2^61), the remaining <= 7 bits feed `hi` (each < 2^38),
// and value() folds lo + hi 2^30 with q = 2^B - c.  A term costs two wide multiplies (8 multiplier-pipe cycles) against three
// wide + one low (14) for a term with its own Shoup quotient estimate, which buys nothing when the factors are this short; the
// result is the canonical residue.
template <class M>
struct WideSum {
    static constexpr int kHiBits = M::kBits - 30;  // 6 or 7
    u64 lo = 0, hi = 0;
    __device__ __forceinline__ void add32(u32 x, u64 w) {
        u32 wl, wh;
        unpack64(w, wl, wh);
        lo = mad_wide(x, wl & 0x3fffffffu, lo);
        hi = mad_wide(x, (wl >> 30) | (wh << 2), hi);
    }
    // x * w for x < 2^8: the product is below 2^45 and goes to `lo` whole                                1 wide + 1 low
    __device__ __forceinline__ void add_small(u32 x, u64 w) {
        u32 wl, wh, al, ah;
        unpack64(w, wl, wh);
        unpack64(mad_wide(x, wl, lo), al, ah);
        lo = pack64(al, mad_lo(x, wh, ah));
    }
    // canonical residue of lo + hi 2^30: with A = floor(lo / 2^B) + floor(hi / 2^(B-30)) < 2^35 the sum is congruent to
    // (lo mod 2^B) + ((hi mod 2^(B-30)) << 30) + A c < 2^54; one more fold leaves < 2^B + 2^35 < 2q          2 wide + 1 low
    __device__ __forceinline__ u64 value() const {
        constexpr u32 c = (u32)M::kC;
        const u64 A = (lo >> M::kBits) + (hi >> kHiBits);
        const u64 base = (lo & M::kMask) + ((hi & ((1u << kHiBits) - 1)) << 30);
        u32 al, ah, yl, yh;
        unpack64(A, al, ah);
        unpack64(mad_wide(al, c, base), yl, yh);
        const u64 Y = pack64(yl, mad_lo(ah, c, yh));
        return csub<M>(mad_wide((u32)(Y >> M::kBits), c, Y & M::kMask), M::q);
    }
};

// pseudo-Mersenne fold: x -> (x mod 2^b) + floor(x / 2^b) * c, congruent to x mod q.
// Result < 2^b + 2^(64-b) * c; one more conditional subtraction is canonical whenever that is < 2q.
template <class M>
__device__ __forceinline__ u64 fold(u64 x) {
    const u64 k = x >> M::kBits;
    return (x & M::kMask) + k * M::kC;
}
// the same when floor(x / 2^b) * c fits 32 bits (one low multiply instead of a 64-bit one)
template <class M>
__device__ __forceinline__ u64 fold_k32(u64 x) {
    const u32 k = (u32)(x >> M::kBits);
    return (x & M::kMask) + (u64)(k * (u32)M::kC);
}
// canonical when floor(x / 2^b) c fits 32 bits: small primes x < 2^50, 61-bit primes any x
template <class M>
__device__ __forceinline__ u64 canon_k32(u64 x) {
    return csub<M>(fold_k32<M>(x), M::q);
}
// canonical residue of x when fold(x) < 2q: small primes x < 2^54 (at 2^55 q1's fold reaches 2^37.5 > 2q), 61-bit primes any x
template <class M>
__device__ __forceinline__ u64 canon(u64 x) {
    return csub<M>(fold<M>(x), M::q);
}

// sum of NP (1 or 2) products x_i * y_i of two VARIABLES (no precomputed quotient), on explicit 32-bit partial products.
// The compiler's lowering of a 128-bit mad.lo.cc.u64 / madc.hi.u64 accumulate and its reduction recomputes partial products
// for the carries and multiplies by zero high words; these issue 6-9 wide multiplies per call instead of 10-16.
//
// 61-bit primes, operands < 2^61, result in [0, 2q).  V = p00 + mid 2^32 + p11 2^64 (mid, p11 accumulate over the
// products in mad.wide chains, no carries).  Quotient Q = qe + floor(qe c / 2^61) with qe ~ floor(V / 2^61) from the
// column tops (low by < 3 + NP), so V - Q q < (4 + NP) q needs only the low 64 bits of V.
template <class M, int NP>
__device__ __forceinline__ u64 mulsum_large(const u64 (&x)[NP], const u64 (&y)[NP]) {
    constexpr u32 c = (u32)M::kC;
    u64 p00[NP], mid = 0, p11 = 0;
#pragma unroll
    for (int i = 0; i < NP; i++) {
        u32 xl, xh, yl, yh;
        unpack64(x[i], xl, xh);
        unpack64(y[i], yl, yh);
        p00[i] = mul_wide(xl, yl);
        mid = i == 0 ? mad_wide(xl, yh, mul_wide(xh, yl)) : mad_wide(xl, yh, mad_wide(xh, yl, mid));
        p11 = i == 0 ? mul_wide(xh, yh) : mad_wide(xh, yh, p11);
    }
    u64 qe = (p11 << 3) + (mid >> 29) + (p00[0] >> 61);
    u64 lo = p00[0];
    if (NP == 2) {
        qe += p00[NP - 1] >> 61;
        lo += p00[NP - 1];  // mod 2^64
    }
    const u64 Q = qe + (mul_wide((u32)(qe >> 32), c) >> 29);
    u32 ll, lh, Ql, Qh, al, ah;
    unpack64(lo, ll, lh);
    lh += (u32)mid;
    unpack64(Q, Ql, Qh);
    unpack64(mad_wide(Ql, c, pack64(ll, lh)), al, ah);
    ah = mad_lo(Qh, c, ah);
    ah -= Ql << 29;
    return fold_k32<M>(pack64(al, ah));
}
// 36/37-bit primes q = 2^B - c, operands < 2^44, result in [0, 2q).  V = p00 + M' 2^32 with M' = mid + p11 2^32 < 2^58;
// M' 2^32 = a_lo 2^32 + a_hi 2^B + b 2^2B  ==  a_lo 2^32 + a_hi c + b c^2, the p00 tops join a_hi, then two folds.
template <class M, int NP>
__device__ __forceinline__ u64 mulsum_small(const u64 (&x)[NP], const u64 (&y)[NP]) {
    constexpr int B = M::kBits;
    constexpr u32 c = (u32)M::kC;
    constexpr u64 c2 = M::kC * M::kC;
    constexpr int sh = 2 * B - 32;
    u64 p00[NP];
    u32 xl[NP], xh[NP], yl[NP], yh[NP], p11 = 0;
#pragma unroll
    for (int i = 0; i < NP; i++) {
        unpack64(x[i], xl[i], xh[i]);
        unpack64(y[i], yl[i], yh[i]);
        p00[i] = mul_wide(xl[i], yl[i]);
        p11 = mad_lo(xh[i], yh[i], p11);
    }
    u64 mp = pack64(0, p11);
#pragma unroll
    for (int i = 0; i < NP; i++) mp = mad_wide(xl[i], yh[i], mad_wide(xh[i], yl[i], mp));
    const u32 b = (u32)(mp >> sh);
    const u64 a = mp & ((1ull << sh) - 1);
    u64 T = (a >> (B - 32)) + (p00[0] >> B);
    u64 S = p00[0] & M::kMask;
    if (NP == 2) {
        T += p00[NP - 1] >> B;
        S += p00[NP - 1] & M::kMask;
    }
    u32 Tl, Th, sl, shi;
    unpack64(T, Tl, Th);
    unpack64(S, sl, shi);
    shi += (u32)a & ((1u << (B - 32)) - 1);
    unpack64(mad_wide(b, (u32)c2, mad_wide(Tl, c, pack64(sl, shi))), sl, shi);
    shi = mad_lo(Th, c, shi);
    shi = mad_lo(b, (u32)(c2 >> 32), shi);
    S = pack64(sl, shi);
    S = mad_wide((u32)(S >> B), c, S & M::kMask);
    return fold_k32<M>(S);
}
template <class M, int NP>
__device__ __forceinline__ u64 mulsum(const u64 (&x)[NP], const u64 (&y)[NP]) {
    if constexpr (M::kSmall)
        return mulsum_small<M, NP>(x, y);
    else
        return mulsum_large<M, NP>(x, y);
}

// x mod q for any 64-bit x (SEAL barrett_reduce_64)
template <class M>
__device__ __forceinline__ u64 reduce64(u64 x) {
    if (!M::kSmall) return canon<M>(x);  // fold(x) <= 2^61 - 1 + 7c < 2q
    u64 r = x - mulhi64(x, M::r1) * M::q;
    return csub<M>(r, M::q);
}

// canonical a*b mod q; operands below 2^44 (36/37-bit primes) or 2^61 (61-bit primes)
template <class M>
__device__ __forceinline__ u64 mulmod(u64 a, u64 b) {
    const u64 xs[1] = {a}, ys[1] = {b};
    return csub<M>(mulsum<M, 1>(xs, ys), M::q);
}

template <class M>
__device__ __forceinline__ u64 addmod(u64 a, u64 b) {
    return csub<M>(a + b, M::q);
}
template <class M>
__device__ __forceinline__ u64 submod(u64 a, u64 b) {
    return a >= b ? a - b : a + M::q - b;
}

}  // namespace fheb
