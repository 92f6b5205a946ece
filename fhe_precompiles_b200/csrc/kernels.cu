// sm_100a kernels for the BFV precompile hot path (add / sub / negate, plain ops, BEHZ multiply,
// relinearisation) and their launchers.  Replaces the SEAL 4.0 Evaluator calls that
// FheApp::run (/root/reference/src/fhe.rs:138-152) triggers for the 36 programs at
// fhe.rs:814-1022.  Integer-pipe work: no tensor cores (SURVEY.md 8d).
//
// Device data layouts (u64 everywhere, limb-major):
//   data-level ciphertext   [poly 0..1][limb q0,q1][4096]                 128 KiB
//   size-3 ciphertext       [poly 0..2][limb q0,q1][4096]
//   BEHZ tensor scratch     [poly 0..2][slot 0..4][4096]                  (already x t; dual words in slots 2..4)
//   key-switch scratch      [poly 0..1][limb q0,q1,P][4096]
//   relin key               [digit 0..1][poly 0..1][limb q0,q1,P][4096]   NTT form, as in the key file
//   plaintext               [4096] u16 coefficients < t, zero padded
#include <atomic>
#include <cstdio>

#include "kernels.h"

namespace fheb {
__constant__ DevTwLow ktl;  // defined before ntt.cuh, which reads it
__constant__ DevConsts kc;  // likewise (modarith.cuh: opaque_zero)
}
#include "ntt.cuh"

namespace fheb {

__constant__ DevTables kt;

cudaError_t upload_constants(const DevConsts &c, const DevTables &t, const DevTwLow &lo) {
    cudaError_t e = cudaMemcpyToSymbol(kc, &c, sizeof(c));
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbol(ktl, &lo, sizeof(lo));
    if (e != cudaSuccess) return e;
    return cudaMemcpyToSymbol(kt, &t, sizeof(t));
}

// =====================================================================================
// K1/K2: batched limb NTT (config 2 microbenchmark; also used by the parity tests)
// =====================================================================================
template <int MI, bool INV>
__device__ __forceinline__ void ntt_limb_body(u64 *limb, u64 *smem, int t) {
    using M = Mod<MI>;
    u64 v[1][8];
    if (!INV) {
        load_natural(limb, v[0], t);
        ntt_forward<M, 1, true, false>(v, smem, kt.twf[MI], t);
        store_chunk8(limb, v[0], t);
    } else {
        load_chunk8(limb, v[0], t);
        ntt_inverse<M, 1, true, false>(v, smem, kt.twi[MI], t, kc.ninv[MI], kc.ninv_w[MI]);
        store_natural(limb, v[0], t);
    }
}

template <bool INV>
// the forward transform fits 40 registers (3 CTAs per SM, +9 % on the 36-bit primes); the inverse does not gain from it
__global__ void __launch_bounds__(kThreads, INV ? 2 : 3) k_ntt(u64 *data, LimbMods mods) {
    extern __shared__ __align__(16) u64 smem[];
    const int t = threadIdx.x;
    u64 *limb = data + (size_t)blockIdx.x * kN;
    switch (mods.mod[blockIdx.x % mods.n]) {
        case MQ0: ntt_limb_body<MQ0, INV>(limb, smem, t); break;
        case MQ1: ntt_limb_body<MQ1, INV>(limb, smem, t); break;
        case MP: ntt_limb_body<MP, INV>(limb, smem, t); break;
        case MB0: ntt_limb_body<MB0, INV>(limb, smem, t); break;
        case MB1: ntt_limb_body<MB1, INV>(limb, smem, t); break;
        default: ntt_limb_body<MSK, INV>(limb, smem, t); break;
    }
}

// =====================================================================================
// K3: ciphertext add / sub / negate   (SEAL add_poly_coeffmod / sub_poly_coeffmod / negate_poly_coeffmod)
// =====================================================================================
template <class M>
__device__ __forceinline__ u64 eltop(u64 a, u64 b, int op) {
    if (op == 0) return addmod<M>(a, b);
    if (op == 1) return submod<M>(a, b);
    return a ? M::q - a : 0;
}
// n2 = number of ulonglong2 elements; limb index = (element / N) & 1
__global__ void __launch_bounds__(256) k_eltwise(const ulonglong2 *__restrict__ a, const ulonglong2 *__restrict__ b,
                                                 ulonglong2 *__restrict__ out, size_t n2, int op) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += stride) {
        ulonglong2 x = a[i];
        ulonglong2 y = (op == 2) ? make_ulonglong2(0, 0) : b[i];
        int limb = (int)((i / (kN / 2)) & 1);
        ulonglong2 r;
        if (limb == 0) {
            r.x = eltop<Mod<MQ0>>(x.x, y.x, op);
            r.y = eltop<Mod<MQ0>>(x.y, y.y, op);
        } else {
            r.x = eltop<Mod<MQ1>>(x.x, y.x, op);
            r.y = eltop<Mod<MQ1>>(x.y, y.y, op);
        }
        out[i] = r;
    }
}

// =====================================================================================
// K4: add_plain / sub_plain (+ optional negate for `pt - ct`)
//     SEAL multiply_add_plain_with_scaling_variant / multiply_sub_plain_with_scaling_variant
// mode bit0: subtract; bit1: negate the whole result afterwards
// =====================================================================================
template <class M>
__device__ __forceinline__ u64 plain_scaled(u64 m, int l) {
    // fix = floor((q mod t) * m + (t+1)/2) / t); scaled = Delta*m + fix mod q_l
    u64 fix = (kc.q_mod_t * m + kc.upper_half_threshold) / kT;
    u64 lo = kc.delta_mod_q[l] * m + fix;  // < 2^36 * 2^12 + small: fits
    return reduce64<M>(lo);
}
__global__ void __launch_bounds__(256) k_plain_addsub(const u64 *__restrict__ ct, const unsigned short *__restrict__ plain,
                                                      u64 *__restrict__ out, size_t n_ops, int mode) {
    size_t total = n_ops * 4 * kN;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        size_t op = i / (4 * kN);
        int rem = (int)(i % (4 * kN));
        int poly = rem / (2 * kN);
        int limb = (rem / kN) & 1;
        int c = rem % kN;
        u64 v = ct[i];
        if (poly == 0) {
            u64 m = plain[op * kN + c];
            if (limb == 0) {
                u64 s = plain_scaled<Mod<MQ0>>(m, 0);
                v = (mode & 1) ? submod<Mod<MQ0>>(v, s) : addmod<Mod<MQ0>>(v, s);
            } else {
                u64 s = plain_scaled<Mod<MQ1>>(m, 1);
                v = (mode & 1) ? submod<Mod<MQ1>>(v, s) : addmod<Mod<MQ1>>(v, s);
            }
        }
        if (mode & 2) v = v ? (limb ? Mod<MQ1>::q : Mod<MQ0>::q) - v : 0;
        out[i] = v;
    }
}

// =====================================================================================
// K5: multiply_plain   (SEAL Evaluator::multiply_plain_normal)
// one CTA per (limb, op): NTT(lift(m)), NTT(c0), NTT(c1), dyadic, 2 x INTT
// =====================================================================================
template <int MI>
__device__ __forceinline__ void mul_plain_body(const u64 *__restrict__ ct, const unsigned short *__restrict__ plain,
                                               u64 *__restrict__ out, u64 *smem, int t) {
    using M = Mod<MI>;
    u64 v[3][8];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        u64 m = plain[r * kThreads + t];
        v[0][r] = m + (m >= kc.upper_half_threshold ? kc.upper_half_incr[MI] : 0);
    }
    load_natural(ct + (size_t)(0 * 2 + MI) * kN, v[1], t);
    load_natural(ct + (size_t)(1 * 2 + MI) * kN, v[2], t);
    ntt_forward<M, 3, true>(v, smem, kt.twf[MI], t);
    u64 d[2][8];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        d[0][r] = mulmod<M>(v[1][r], v[0][r]);
        d[1][r] = mulmod<M>(v[2][r], v[0][r]);
    }
    ntt_inverse<M, 2>(d, smem, kt.twi[MI], t, kc.ninv[MI], kc.ninv_w[MI]);
    store_natural(out + (size_t)(0 * 2 + MI) * kN, d[0], t);
    store_natural(out + (size_t)(1 * 2 + MI) * kN, d[1], t);
}
__global__ void __launch_bounds__(kThreads, 1) k_mul_plain(const u64 *__restrict__ ct, const unsigned short *__restrict__ plain,
                                                            u64 *__restrict__ out) {
    extern __shared__ __align__(16) u64 smem[];
    const size_t op = blockIdx.y;
    const u64 *c = ct + op * 4 * kN;
    const unsigned short *p = plain + op * kN;
    u64 *o = out + op * 4 * kN;
    if (blockIdx.x == 0)
        mul_plain_body<MQ0>(c, p, o, smem, threadIdx.x);
    else
        mul_plain_body<MQ1>(c, p, o, smem, threadIdx.x);
}

// =====================================================================================
// K6-K8: BEHZ multiply   (SEAL Evaluator::bfv_multiply steps (1)-(6); RNSTool::fastbconv_m_tilde, sm_mrq, fast_floor,
// fastbconv_sk) on the DUAL base (params.h kDualPrime, devconsts.h d_*).  bfv_multiply's result is a function of integer
// polynomials -- the extended operands a' = (y0 + r q) / m~, their product D, f = (t D - y0') / q -- and does not depend on the
// auxiliary primes that carry them, so they are carried by six primes below 2^30, two per 64-bit word, where a butterfly costs
// one IMAD.HI + two IMAD per lane (8 multiplier cycles per 30 bits) instead of 6 IMAD.WIDE + 4 IMAD (32 cycles per 61 bits
// on SEAL's Bsk primes).  The dual words live in slots e = 2..4 of the 5-limb scratch arrays (engine.h ScratchMap).
//   k_ext_conv_d     : a' mod s_i for the 4 input polynomials                         eltwise
//   k_ext_ntt_d      : 12 forward dual transforms, in place                           grid (12, ops)
//   k_tensor_intt_d  : dyadic tensor + 9 inverse dual transforms (x N^-1 t)           grid (9, ops)
//   k_floor_sk_d     : exact CRT of t D -> t_l -> y0 -> f on (s_0..s_3) -> f mod q_l   eltwise
//   k_tensor_floor_d : k_tensor_intt_d + k_floor_sk_d in one kernel (chunks >= 96 ops) grid (3, ops)
// =====================================================================================
// y0 = t0 q1 + t1 q0 as a 128-bit integer (t_l canonical residues mod q_l): q_l = 2^36 - c_l, so
// y0 = ((t0 + t1) << 36) - (t0 c1 + t1 c0), one multiply chain and a shift.  Shared by k_ext_conv_d and k_floor_sk_d.
__device__ __forceinline__ void punctured_sum(u64 t0, u64 t1, u64 &ylo, u64 &yhi) {
    constexpr u32 c0 = (u32)Mod<MQ0>::kC, c1 = (u32)Mod<MQ1>::kC;
    u32 t0l, t0h, t1l, t1h, pl, ph;
    unpack64(t0, t0l, t0h);
    unpack64(t1, t1l, t1h);
    unpack64(mad_wide(t0l, c1, mul_wide(t1l, c0)), pl, ph);
    ph = mad_lo(t0h, c1, ph);  // t_h < 16
    ph = mad_lo(t1h, c0, ph);
    const u64 pv = pack64(pl, ph);  // t0 c1 + t1 c0 < 2^56
    const u64 ts = t0 + t1, sh = ts << 36;
    ylo = sh - pv;
    yhi = (ts >> 28) - (sh < pv ? 1 : 0);
}
// Base extension in the integer domain.  SEAL's fastbconv_m_tilde + sm_mrq compute, per auxiliary prime p, (y0 + r q) m~^-1
// mod p with r = -y0 q^-1 mod m~ centred: y0 + r q is an exact multiple of m~ = 2^32, so the value is the INTEGER
// Z = (y0 + r q) / 2^32 (|Z| < 2^72) reduced mod p.  ext_shared forms Z once per coefficient, as base + m 2^61 (- q if neg);
// ext_dual reduces it mod each dual prime.
__device__ __forceinline__ void ext_shared(u64 x0, u64 x1, u64 &base, u32 &m, bool &neg) {
    const u64 t0 = shoup<Mod<MQ0>>(x0, kc.ext_in[0].w, kc.ext_in[0].ws);
    const u64 t1 = shoup<Mod<MQ1>>(x1, kc.ext_in[1].w, kc.ext_in[1].ws);
    u64 ylo, yhi;
    punctured_sum(t0, t1, ylo, yhi);
    const u32 ymt = (u32)ylo;
    const u32 rm = ymt * kc.neg_inv_q_mod_mtilde;
    neg = rm >= 0x80000000u;
    // (y0 + rm q) >> 32 = A + rm q_w1 + (rm q_w2 << 32); the low words of y0 and rm q_w0 cancel (carry iff non-zero)
    const u64 A = ((ylo >> 32) | (yhi << 32)) + (mul_wide(rm, kc.q_w[0]) >> 32) + (ymt != 0 ? 1 : 0);
    const u64 Bv = mul_wide(rm, kc.q_w[1]), Cv = mul_wide(rm, kc.q_w[2]);
    const u64 sAB = A + Bv;
    m = (u32)(sAB >> 61) + (sAB < A ? 8u : 0u) + (u32)(Cv >> 29);             // < 2^12
    base = (sAB & ((1ull << 61) - 1)) + ((Cv & ((1ull << 29) - 1)) << 32);  // < 2^62
}

template <int D>
__device__ __forceinline__ u64 ext_dual(u64 base, u32 m, bool neg) {
    u32 bl, bh, r[2];
    unpack64(base, bl, bh);
#pragma unroll
    for (int lane = 0; lane < 2; lane++) {
        const int i = 2 * D + lane;
        const u32 s = lane ? ModDual<D>::s1 : ModDual<D>::s0;
        // Z = base + m 2^61 (- q)  ==  base_lo + base_hi R32 + m R61 (+ NQ)   < 2^61
        u64 V = mad_wide(bh, kc.d_R32[i], (u64)bl);
        V = mad_wide(m, kc.d_R61[i], V) + (neg ? kc.d_NQ[i] : 0u);
        r[lane] = barrett61(V, kc.d_mu61[i], s);  // [0, 4s): the forward transform's input range
    }
    return pack64(r[0], r[1]);
}
// The extension is its own full-occupancy elementwise kernel: the shared part is computed once per coefficient (a CTA per dual
// word would redo it three times) and the residues are left, coefficient domain, in the scratch slots that k_ext_ntt_d then
// transforms in place with 40 registers, 3 CTAs per SM.
__global__ void __launch_bounds__(256) k_ext_conv_d(const u64 *__restrict__ a, const u64 *__restrict__ b, u64 *__restrict__ nttbuf,
                                                    size_t n_ops) {
    const size_t total = n_ops * 4 * (kN / 2);
    for (size_t g = (size_t)blockIdx.x * 256 + threadIdx.x; g < total; g += (size_t)gridDim.x * 256) {
        const size_t op = g / (4 * (kN / 2));
        const int p = (int)((g / (kN / 2)) & 3), i = 2 * (int)(g & (kN / 2 - 1));
        const u64 *ct = (p < 2 ? a : b) + op * 4 * kN + (size_t)(p & 1) * 2 * kN;
        const ulonglong2 x0 = *reinterpret_cast<const ulonglong2 *>(ct + i), x1 = *reinterpret_cast<const ulonglong2 *>(ct + kN + i);
        u64 base0, base1;
        u32 m0, m1;
        bool neg0, neg1;
        ext_shared(x0.x, x1.x, base0, m0, neg0);
        ext_shared(x0.y, x1.y, base1, m1, neg1);
        u64 *dst = nttbuf + (op * 20 + (size_t)p * 5 + 2) * kN + i;
        *reinterpret_cast<ulonglong2 *>(dst) = make_ulonglong2(ext_dual<0>(base0, m0, neg0), ext_dual<0>(base1, m1, neg1));
        *reinterpret_cast<ulonglong2 *>(dst + kN) = make_ulonglong2(ext_dual<1>(base0, m0, neg0), ext_dual<1>(base1, m1, neg1));
        *reinterpret_cast<ulonglong2 *>(dst + 2 * kN) = make_ulonglong2(ext_dual<2>(base0, m0, neg0), ext_dual<2>(base1, m1, neg1));
    }
}
template <int D>
__device__ __forceinline__ void ntt_dual_body(u64 *__restrict__ limb, u64 *smem, int t) {
    using M = ModDual<D>;
    u64 v[1][8];
    load_natural(limb, v[0], t);
    ntt_forward<M, 1, false, false>(v, smem, kt.twf[M::kIndex], t);  // values stay in [0, 4s)
    store_chunk8_lm(limb, v[0], t);
}
__global__ void __launch_bounds__(kThreads, 3) k_ext_ntt_d(u64 *__restrict__ nttbuf) {
    extern __shared__ __align__(16) u64 smem[];
    const size_t op = blockIdx.y;
    const int p = blockIdx.x / 3, d = blockIdx.x % 3;
    u64 *limb = nttbuf + (op * 20 + (size_t)(p * 5 + 2 + d)) * kN;
    const int t = threadIdx.x;
    switch (d) {
        case 0: ntt_dual_body<0>(limb, smem, t); break;
        case 1: ntt_dual_body<1>(limb, smem, t); break;
        default: ntt_dual_body<2>(limb, smem, t); break;
    }
}
// the dyadic tensor of dual word D for output polynomial d + its inverse transform, left in registers (lanes in [0, 2s))
template <int D, bool kTrailSync>
__device__ __forceinline__ void tensor_intt_dual_regs(const u64 *__restrict__ nb, int d, u64 (&v)[1][8], u64 *smem, int t) {
    using M = ModDual<D>;
    constexpr int E = 2 + D;
    const u64 *a0 = nb + (size_t)(0 * 5 + E) * kN, *a1 = nb + (size_t)(1 * 5 + E) * kN;
    const u64 *b0 = nb + (size_t)(2 * 5 + E) * kN, *b1 = nb + (size_t)(3 * 5 + E) * kN;
    const u32 mu0 = kc.d_mu61[2 * D], mu1 = kc.d_mu61[2 * D + 1];
    const ulonglong2 *pa0 = lm_ptr(a0, t), *pa1 = lm_ptr(a1, t), *pb0 = lm_ptr(b0, t), *pb1 = lm_ptr(b1, t);  // pair r at [r * kLm]
    auto one = [&](u64 x0, u64 y0) -> u64 {
        u32 xl, xh, yl, yh;
        unpack64(x0, xl, xh);
        unpack64(y0, yl, yh);
        const u32 xs0[1] = {xl}, ys0[1] = {yl}, xs1[1] = {xh}, ys1[1] = {yh};
        return pack64(dual_mulsum<1>(xs0, ys0, M::s0, mu0), dual_mulsum<1>(xs1, ys1, M::s1, mu1));
    };
    auto two = [&](u64 x0, u64 y0, u64 x1, u64 y1) -> u64 {
        u32 al, ah, bl, bh, cl, ch, dl, dh;
        unpack64(x0, al, ah);
        unpack64(y0, bl, bh);
        unpack64(x1, cl, ch);
        unpack64(y1, dl, dh);
        const u32 xs0[2] = {al, cl}, ys0[2] = {bl, dl}, xs1[2] = {ah, ch}, ys1[2] = {bh, dh};
        return pack64(dual_mulsum<2>(xs0, ys0, M::s0, mu0), dual_mulsum<2>(xs1, ys1, M::s1, mu1));
    };
    if (d == 1) {
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const ulonglong2 x0 = pa0[r * kLm], y1 = pb1[r * kLm], x1 = pa1[r * kLm], y0 = pb0[r * kLm];
            v[0][2 * r] = two(x0.x, y1.x, x1.x, y0.x);
            v[0][2 * r + 1] = two(x0.y, y1.y, x1.y, y0.y);
        }
    } else {
        const ulonglong2 *px = d == 0 ? pa0 : pa1, *py = d == 0 ? pb0 : pb1;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const ulonglong2 x = px[r * kLm], y = py[r * kLm];
            v[0][2 * r] = one(x.x, y.x);
            v[0][2 * r + 1] = one(x.y, y.y);
        }
    }
    ntt_inverse<M, 1, false, kTrailSync>(v, smem, kt.twi[M::kIndex], t, kc.d_ninv_t[D], kc.d_ninv_t_w[D]);  // [0, 2s)
}
template <int D>
__device__ __forceinline__ void tensor_intt_dual_body(const u64 *__restrict__ nb, int d, u64 *__restrict__ dst, u64 *smem, int t) {
    u64 v[1][8];
    tensor_intt_dual_regs<D, false>(nb, d, v, smem, t);
    store_natural(dst, v[0], t);
}
__global__ void __launch_bounds__(kThreads, 3) k_tensor_intt_d(const u64 *__restrict__ nttbuf, u64 *__restrict__ tens) {
    extern __shared__ __align__(16) u64 smem[];
    const size_t op = blockIdx.y;
    const int d = blockIdx.x / 3, e = blockIdx.x % 3;
    const u64 *nb = nttbuf + op * 20 * kN;
    u64 *dst = tens + (op * 15 + (size_t)(d * 5 + 2 + e)) * kN;
    const int t = threadIdx.x;
    switch (e) {
        case 0: tensor_intt_dual_body<0>(nb, d, dst, smem, t); break;
        case 1: tensor_intt_dual_body<1>(nb, d, dst, smem, t); break;
        default: tensor_intt_dual_body<2>(nb, d, dst, smem, t); break;
    }
}
__device__ __forceinline__ u32 dual_prime(int i) {
    constexpr u32 p[6] = {kDualPrime[0], kDualPrime[1], kDualPrime[2], kDualPrime[3], kDualPrime[4], kDualPrime[5]};
    return p[i];
}
// per coefficient: the three dual words of t D (each lane in [0, 2s))  ->  limbs q0, q1 of the size-3 product
__device__ __forceinline__ void floor_sk_coeff_d(u64 w0, u64 w1, u64 w2, u64 &o0, u64 &o1) {
    using Q0 = Mod<MQ0>;
    using Q1 = Mod<MQ1>;
    u32 r[6], y[6];
    unpack64(w0, r[0], r[1]);
    unpack64(w1, r[2], r[3]);
    unpack64(w2, r[4], r[5]);
    // v = round(sum y_i / s_i): every s_i is within 2^-12 of 2^30, so y_i / 2^30 (in units of 2^-16: y_i >> 14) is off by
    // less than 2^-11 per term -- far inside the 1/2 - 2^-13 that the rounding tolerates (|t D| / S < 2^-13)
    u32 est = 1u << 15;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        y[i] = shoup32(r[i], kc.d_C[i], kc.d_Cs[i], dual_prime(i));  // [(S/s_i)^-1 r_i] in [0, 2s)
        est += y[i] >> 14;
    }
    const u32 v = est >> 16;  // t D = sum y_i (S/s_i) - v S exactly
    u64 t0, t1;
    {
        WideSum<Q0> s;  // exact sum of the six products + v KN, one reduction (modarith.cuh)
#pragma unroll
        for (int i = 0; i < 6; i++) s.add32(y[i], kc.d_K[i][0].w);
        s.add_small(v, kc.d_KN[0]);
        t0 = s.value();
    }
    {
        WideSum<Q1> s;
#pragma unroll
        for (int i = 0; i < 6; i++) s.add32(y[i], kc.d_K[i][1].w);
        s.add_small(v, kc.d_KN[1]);
        t1 = s.value();
    }
    // fast_floor: y0 = t0 q1 + t1 q0 (the q-part of t D with its fast-base-conversion overflow), f = (t D - y0) / q on s_0..s_3
    u64 ylo, yhi;
    punctured_sum(t0, t1, ylo, yhi);
    const u32 u2 = (u32)((ylo >> 58) | (yhi << 6));  // y0 < 2^73
    const u64 low58 = ylo & ((1ull << 58) - 1);
    u32 tb[4], est2 = 1u << 15;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const u32 s = dual_prime(i);
        const u32 yi = csub32(barrett61(mad_wide(u2, kc.d_R58[i], low58), kc.d_mu61[i], s), 2 * s);  // y0 mod s_i in [0, 2s)
        tb[i] = shoup32(r[i] + 2 * s - yi, kc.d_W[i], kc.d_Ws[i], s);                               // [f (S4/s_i)^-1] in [0, 2s)
        est2 += tb[i] >> 14;
    }
    const u32 vp = est2 >> 16;  // f = sum tb_i (S4/s_i) - v' S4 exactly (|f| / S4 < 2^-24)
    {
        WideSum<Q0> s;
#pragma unroll
        for (int i = 0; i < 4; i++) s.add32(tb[i], kc.d_P[i][0].w);
        s.add_small(vp, kc.d_NS4[0]);
        o0 = s.value();
    }
    {
        WideSum<Q1> s;
#pragma unroll
        for (int i = 0; i < 4; i++) s.add32(tb[i], kc.d_P[i][1].w);
        s.add_small(vp, kc.d_NS4[1]);
        o1 = s.value();
    }
}
__global__ void __launch_bounds__(256, 3) k_floor_sk_d(const u64 *__restrict__ tens, u64 *__restrict__ c3, size_t n_ops) {
    const size_t total = n_ops * 3 * (kN / 2);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += stride) {
        const size_t opp = g / (kN / 2);  // op*3 + poly
        const int i = 2 * (int)(g % (kN / 2));
        const ulonglong2 *in = reinterpret_cast<const ulonglong2 *>(tens + opp * 5 * kN + i);
        const ulonglong2 w0 = in[2 * (kN / 2)], w1 = in[3 * (kN / 2)], w2 = in[4 * (kN / 2)];
        u64 ax, ay, bx, by;
        floor_sk_coeff_d(w0.x, w1.x, w2.x, ax, bx);
        floor_sk_coeff_d(w0.y, w1.y, w2.y, ay, by);
        ulonglong2 *out = reinterpret_cast<ulonglong2 *>(c3 + opp * 2 * kN + i);
        out[0] = make_ulonglong2(ax, ay);
        out[kN / 2] = make_ulonglong2(bx, by);
    }
}

// ---- K7d + K8d in one kernel (chunks >= 96 ops; smaller ones run the two kernels above): one CTA per (output polynomial d, op) runs the three
// dual words one after the other -- dyadic tensor, inverse transform -- parks the first two results at each thread's own eight
// slots in shared memory (r * 512 + t: the coefficients it owns after every inverse transform) and finishes with
// floor_sk_coeff_d on its eight coefficients, so the tensor product never goes through HBM (0.59 MB per op less DRAM traffic:
// the batch runs into the board's power limit, where bytes not moved are clock).  Same structure as k_ks_tail_ksd: 2 CTAs per SM.
__global__ void __launch_bounds__(kThreads, 2) k_tensor_floor_d(const u64 *__restrict__ nttbuf, u64 *__restrict__ c3) {
    extern __shared__ __align__(16) u64 smem[];  // [3][kN]: exchange buffer, word 0, word 1
    const size_t op = blockIdx.y;
    const int d = blockIdx.x, t = threadIdx.x;
    const u64 *nb = nttbuf + op * 20 * kN;
    u64 *park0 = smem + kN, *park1 = smem + 2 * kN;
    {
        u64 v[1][8];
        tensor_intt_dual_regs<0, true>(nb, d, v, smem, t);
#pragma unroll
        for (int r = 0; r < 8; r++) park0[r * kThreads + t] = v[0][r];
    }
    {
        u64 v[1][8];
        tensor_intt_dual_regs<1, true>(nb, d, v, smem, t);
#pragma unroll
        for (int r = 0; r < 8; r++) park1[r * kThreads + t] = v[0][r];
    }
    u64 v[1][8];
    tensor_intt_dual_regs<2, false>(nb, d, v, smem, t);
    u64 *out = c3 + (op * 3 + d) * 2 * kN;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        u64 o0, o1;
        floor_sk_coeff_d(park0[r * kThreads + t], park1[r * kThreads + t], v[0][r], o0, o1);
        out[r * kThreads + t] = o0;
        out[kN + r * kThreads + t] = o1;
    }
}

// =====================================================================================
// K9: key switching  (SEAL Evaluator::switch_key_inplace, BFV branch) on SEAL's key primes q0, q1, P, for chunks < 96 ops
//   k_digit_ntt    : NTT_J([c2]_I)                       grid (6 = I*3+J, ops)   -> dig [op][2][3][N]
//   k_ks_intt      : INTT_J(sum_I dig[I][J] * rk[I][k][J]) grid (6 = k*3+J, ops) -> ks  [op][2][3][N]
//   k_relin_finish : rounded division by P, added to (c0, c1)   (K9b below)
// =====================================================================================
template <int MI>
__device__ __forceinline__ void digit_ntt_body(const u64 *__restrict__ src, u64 *__restrict__ dst, u64 *smem, int t) {
    using M = Mod<MI>;
    u64 v[1][8];
    load_natural(src, v[0], t);
    ntt_forward<M, 1, false, false>(v, smem, kt.twf[MI], t);  // lazy (< 2^43): the key MAC reduces a 128-bit sum anyway
    store_chunk8_lm(dst, v[0], t);
}
__global__ void __launch_bounds__(kThreads, 3) k_digit_ntt(const u64 *__restrict__ c3, u64 *__restrict__ dig) {
    extern __shared__ __align__(16) u64 smem[];
    const size_t op = blockIdx.y;
    const int I = blockIdx.x / 3, J = blockIdx.x % 3;
    const u64 *src = c3 + op * 6 * kN + 4 * kN + (size_t)I * kN;
    u64 *dst = dig + (op * 6 + blockIdx.x) * kN;
    const int t = threadIdx.x;
    switch (J) {
        case 0: digit_ntt_body<MQ0>(src, dst, smem, t); break;
        case 1: digit_ntt_body<MQ1>(src, dst, smem, t); break;
        default: digit_ntt_body<MP>(src, dst, smem, t); break;
    }
}

template <int MI>
__device__ __forceinline__ void ks_intt_body(const u64 *__restrict__ dg, const u64 *__restrict__ rk, int k, u64 *__restrict__ dst,
                                             u64 *smem, int t) {
    using M = Mod<MI>;
    u64 d0[8], d1[8], k0[8], k1[8];
    load_chunk8_lm(dg + (size_t)(0 * 3 + MI) * kN, d0, t);
    load_chunk8_lm(dg + (size_t)(1 * 3 + MI) * kN, d1, t);
    load_chunk8_ldg(rk + (size_t)((0 * 2 + k) * 3 + MI) * kN, k0, t);
    load_chunk8_ldg(rk + (size_t)((1 * 2 + k) * 3 + MI) * kN, k1, t);
    u64 v[1][8];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const u64 xs[2] = {d0[r], d1[r]}, ys[2] = {k0[r], k1[r]};  // digits lazy (< 2^43), key canonical
        v[0][r] = mulsum<M, 2>(xs, ys);
    }
    ntt_inverse<M, 1, true, false>(v, smem, kt.twi[MI], t, kc.ninv[MI], kc.ninv_w[MI]);
    store_natural(dst, v[0], t);
}
// rk: every op's key, or (key_index non-null) op i reads the key rks[key_index[i]]
__global__ void __launch_bounds__(kThreads, 2) k_ks_intt(const u64 *__restrict__ dig, const u64 *__restrict__ rk,
                                                          const u64 *const *__restrict__ rks, const int *__restrict__ key_index,
                                                          u64 *__restrict__ ks) {
    extern __shared__ __align__(16) u64 smem[];
    const size_t op = blockIdx.y;
    const int k = blockIdx.x / 3, J = blockIdx.x % 3;
    if (key_index) rk = rks[key_index[op]];
    const u64 *dg = dig + op * 6 * kN;
    u64 *dst = ks + (op * 6 + blockIdx.x) * kN;
    const int t = threadIdx.x;
    switch (J) {
        case 0: ks_intt_body<MQ0>(dg, rk, k, dst, smem, t); break;
        case 1: ks_intt_body<MQ1>(dg, rk, k, dst, smem, t); break;
        default: ks_intt_body<MP>(dg, rk, k, dst, smem, t); break;
    }
}

// =====================================================================================
// K9d: the key switch on the dual base, for chunks >= 96 ops (+3 % over SEAL's three key primes, DESIGN.md section 8).  switch_key_inplace's sums S_km = sum_j d_j * rk_jkm mod m are the
// residues of ONE integer polynomial per output k: U_k = sum_j d_j * RK_jk with the key lifted to integers RK == rk (mod q0, q1,
// P), 0 <= RK < 3 Q.  |U_k| < 2 N 2^36 2^111 = 2^160 << S / 2, so U_k is carried exactly by the six dual primes: 6 forward + 6
// inverse DUAL transforms instead of 6 + 6 on 36/37-bit primes, and U_k mod (q0, q1, P) follows by the same CRT-with-rounding
// as in k_floor_sk_d.  Same bits as SEAL (the oracle follows SEAL; prototyped in Python first).
//   k_rk_intt_ksd / k_rk_lift_ksd / k_rk_ntt_ksd : the key -> coefficient form -> integer lift mod s_i -> dual NTT (per call;
//                     K keys in the same three launches, key-major: [K][12][N] at each stage)
//   k_digit_ntt_ksd : dual NTT of the two digits ([c2]_{q_j} as integers)          grid (6 = j*3+w, ops) -> dig [op][2][3][N]
//   k_ks_tail_ksd   : MAC with the lifted key + inverse dual NTTs, U mod (P, q0, q1), rounded division by P, add to (c0, c1)
//                     grid (2 = k, ops) -> out [op][2][2][N]
// =====================================================================================
template <int MI>
__device__ __forceinline__ void rk_intt_body(const u64 *__restrict__ src, u64 *__restrict__ dst, u64 *smem, int t) {
    using M = Mod<MI>;
    u64 v[1][8];
    load_chunk8_ldg(src, v[0], t);
    ntt_inverse<M, 1, true, false>(v, smem, kt.twi[MI], t, kc.ninv[MI], kc.ninv_w[MI]);
    store_natural(dst, v[0], t);
}
// grid (12 limbs, K keys): key y is rk itself (K = 1, rks null) or rks[y]
__global__ void __launch_bounds__(kThreads, 2) k_rk_intt_ksd(const u64 *__restrict__ rk, const u64 *const *__restrict__ rks,
                                                              u64 *__restrict__ coef) {
    extern __shared__ __align__(16) u64 smem[];
    const int limb = blockIdx.x, t = threadIdx.x;
    if (rks) rk = rks[blockIdx.y];
    coef += (size_t)blockIdx.y * 12 * kN;
    switch (limb % 3) {
        case 0: rk_intt_body<MQ0>(rk + (size_t)limb * kN, coef + (size_t)limb * kN, smem, t); break;
        case 1: rk_intt_body<MQ1>(rk + (size_t)limb * kN, coef + (size_t)limb * kN, smem, t); break;
        default: rk_intt_body<MP>(rk + (size_t)limb * kN, coef + (size_t)limb * kN, smem, t); break;
    }
}
// coef [K][4 = j*2+k][3 moduli][N] -> lifted [K][4][3 dual words][N], every lane in [0, 4s)
__global__ void __launch_bounds__(256) k_rk_lift_ksd(const u64 *__restrict__ coef, u64 *__restrict__ lifted) {
    const int g = blockIdx.x * 256 + threadIdx.x;  // K * 4 * N threads
    const int jk = g / kN, i = g % kN;
    const u64 *c = coef + (size_t)jk * 3 * kN + i;
    const u64 y[3] = {shoup<Mod<MQ0>>(c[0], kc.lk_C[0].w, kc.lk_C[0].ws), shoup<Mod<MQ1>>(c[kN], kc.lk_C[1].w, kc.lk_C[1].ws),
                      shoup<Mod<MP>>(c[2 * kN], kc.lk_C[2].w, kc.lk_C[2].ws)};
    u32 lane[6];
#pragma unroll
    for (int l = 0; l < 6; l++) {
        const u32 s = dual_prime(l);
        u32 acc = 0;
#pragma unroll
        for (int m = 0; m < 3; m++) {
            const u32 ym = barrett61(y[m], kc.d_mu61[l], s);                                    // y_m mod s_l, [0, 4s)
            acc = csub32(acc, 2 * s) + shoup32(ym, kc.lk_R[m][l], kc.lk_Rs[m][l], s);           // < 2s + 2s
        }
        lane[l] = acc;
    }
    u64 *o = lifted + (size_t)jk * 3 * kN + i;
    o[0] = pack64(lane[0], lane[1]);
    o[kN] = pack64(lane[2], lane[3]);
    o[2 * kN] = pack64(lane[4], lane[5]);
}
// grid 12 K: limb x of key x / 12
__global__ void __launch_bounds__(kThreads, 3) k_rk_ntt_ksd(const u64 *__restrict__ lifted, u64 *__restrict__ rkd) {
    extern __shared__ __align__(16) u64 smem[];
    const int limb = blockIdx.x, t = threadIdx.x;
    u64 v[1][8];
    load_natural(lifted + (size_t)limb * kN, v[0], t);
    switch (limb % 3) {
        case 0: ntt_forward<ModDual<0>, 1, false, false>(v, smem, kt.twf[kNumMod + 0], t); break;
        case 1: ntt_forward<ModDual<1>, 1, false, false>(v, smem, kt.twf[kNumMod + 1], t); break;
        default: ntt_forward<ModDual<2>, 1, false, false>(v, smem, kt.twf[kNumMod + 2], t); break;
    }
    store_chunk8_lm(rkd + (size_t)limb * kN, v[0], t);
}
template <int D>
__device__ __forceinline__ void digit_ntt_ksd_body(const u64 *__restrict__ src, u64 *__restrict__ dst, u64 *smem, int t) {
    using M = ModDual<D>;
    u64 v[1][8];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const u64 x = src[r * kThreads + t];  // < 2^36
        v[0][r] = pack64(barrett61(x, kc.d_mu61[2 * D], M::s0), barrett61(x, kc.d_mu61[2 * D + 1], M::s1));
    }
    ntt_forward<M, 1, false, false>(v, smem, kt.twf[M::kIndex], t);
    store_chunk8_lm(dst, v[0], t);
}
__global__ void __launch_bounds__(kThreads, 3) k_digit_ntt_ksd(const u64 *__restrict__ c3, u64 *__restrict__ dig) {
    extern __shared__ __align__(16) u64 smem[];
    const size_t op = blockIdx.y;
    const int j = blockIdx.x / 3, w = blockIdx.x % 3;
    const u64 *src = c3 + op * 6 * kN + 4 * kN + (size_t)j * kN;
    u64 *dst = dig + (op * 6 + blockIdx.x) * kN;
    const int t = threadIdx.x;
    switch (w) {
        case 0: digit_ntt_ksd_body<0>(src, dst, smem, t); break;
        case 1: digit_ntt_ksd_body<1>(src, dst, smem, t); break;
        default: digit_ntt_ksd_body<2>(src, dst, smem, t); break;
    }
}
template <int D, bool kTrailSync>
__device__ __forceinline__ void ks_intt_ksd_regs(const u64 *__restrict__ dg, const u64 *__restrict__ rkd, int k, u64 (&v)[1][8], u64 *smem,
                                                 int t) {
    using M = ModDual<D>;
    const u32 mu0 = kc.d_mu61[2 * D], mu1 = kc.d_mu61[2 * D + 1];
    const ulonglong2 *pd0 = lm_ptr(dg + (size_t)(0 * 3 + D) * kN, t), *pd1 = lm_ptr(dg + (size_t)(1 * 3 + D) * kN, t);
    const ulonglong2 *pk0 = lm_ptr(rkd + (size_t)((0 * 2 + k) * 3 + D) * kN, t), *pk1 = lm_ptr(rkd + (size_t)((1 * 2 + k) * 3 + D) * kN, t);
    auto mac = [&](u64 x0, u64 y0, u64 x1, u64 y1) -> u64 {
        u32 al, ah, bl, bh, cl, ch, dl, dh;
        unpack64(x0, al, ah);
        unpack64(y0, bl, bh);
        unpack64(x1, cl, ch);
        unpack64(y1, dl, dh);
        const u32 xs0[2] = {al, cl}, ys0[2] = {bl, dl}, xs1[2] = {ah, ch}, ys1[2] = {bh, dh};
        return pack64(dual_mulsum<2>(xs0, ys0, M::s0, mu0), dual_mulsum<2>(xs1, ys1, M::s1, mu1));
    };
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const ulonglong2 x0 = pd0[r * kLm], x1 = pd1[r * kLm], y0 = __ldg(pk0 + r * kLm), y1 = __ldg(pk1 + r * kLm);
        v[0][2 * r] = mac(x0.x, y0.x, x1.x, y1.x);
        v[0][2 * r + 1] = mac(x0.y, y0.y, x1.y, y1.y);
    }
    ntt_inverse<M, 1, false, kTrailSync>(v, smem, kt.twi[M::kIndex], t, kc.d_ninv[D], kc.d_ninv_w[D]);  // [0, 2s)
}
// one coefficient: the three dual words of U_k (lanes in [0, 2s)), c3's limbs -> the two output limbs
__device__ __forceinline__ void ks_finish_coeff_ksd(u64 w0, u64 w1, u64 w2, u64 c0, u64 c1, u64 &o0, u64 &o1) {
    using Q0 = Mod<MQ0>;
    using Q1 = Mod<MQ1>;
    using PP = Mod<MP>;
    u32 r[6], y[6];
    unpack64(w0, r[0], r[1]);
    unpack64(w1, r[2], r[3]);
    unpack64(w2, r[4], r[5]);
    u32 est = 1u << 15;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        y[i] = shoup32(r[i], kc.d_C[i], kc.d_Cs[i], dual_prime(i));
        est += y[i] >> 14;
    }
    const u32 v = est >> 16;  // U = sum y_i (S/s_i) - v S exactly (|U| / S < 2^-19)
    u64 sp;
    {
        WideSum<PP> s;
#pragma unroll
        for (int i = 0; i < 6; i++) s.add32(y[i], kc.ksK[i][2].w);
        s.add_small(v, kc.ksKN[2]);
        sp = s.value();
    }
    // RNSTool::divide_and_round_q_last with its multiplication by P^-1 folded into the sums (devconsts.h ksKd ...):
    //   out_l = c_l + (U - (last - P/2)) P^-1 mod q_l,  last = (U mod P + P/2) mod P < 2^37 split at bit 30
    const u64 last = csub<PP>(sp + kc.half_P, PP::q);
    const u32 last_lo = (u32)last & 0x3fffffffu, last_hi = (u32)(last >> 30);
    {
        WideSum<Q0> s;  // seven products below 2^61 + small terms: < 2^64
#pragma unroll
        for (int i = 0; i < 6; i++) s.add32(y[i], kc.ksKd[i][0]);
        s.add32(last_lo, kc.ksNd[0]);
        s.add_small(v, kc.ksKNd[0]);
        s.add_small(last_hi, kc.ksNd30[0]);
        s.lo += c0 + kc.ksHd[0];
        o0 = s.value();
    }
    {
        WideSum<Q1> s;
#pragma unroll
        for (int i = 0; i < 6; i++) s.add32(y[i], kc.ksKd[i][1]);
        s.add32(last_lo, kc.ksNd[1]);
        s.add_small(v, kc.ksKNd[1]);
        s.add_small(last_hi, kc.ksNd30[1]);
        s.lo += c1 + kc.ksHd[1];
        o1 = s.value();
    }
}

// ---- the tail of the key switch in one kernel: one CTA per (output polynomial k, op), the three dual
// words of U_k one after the other with the first two parked in shared memory (as k_tensor_floor_d): U_k never goes through HBM.
// rkd: the prepared key of every op, or (key_index non-null) [K][12][N] with op i under key key_index[i]
__global__ void __launch_bounds__(kThreads, 2) k_ks_tail_ksd(const u64 *__restrict__ dig, const u64 *__restrict__ rkd,
                                                              const int *__restrict__ key_index, const u64 *__restrict__ c3,
                                                              u64 *__restrict__ out) {
    extern __shared__ __align__(16) u64 smem[];  // [3][kN]
    const size_t op = blockIdx.y;
    const int k = blockIdx.x, t = threadIdx.x;
    if (key_index) rkd += (size_t)key_index[op] * 12 * kN;
    const u64 *dg = dig + op * 6 * kN;
    u64 *park0 = smem + kN, *park1 = smem + 2 * kN;
    {
        u64 v[1][8];
        ks_intt_ksd_regs<0, true>(dg, rkd, k, v, smem, t);
#pragma unroll
        for (int r = 0; r < 8; r++) park0[r * kThreads + t] = v[0][r];
    }
    {
        u64 v[1][8];
        ks_intt_ksd_regs<1, true>(dg, rkd, k, v, smem, t);
#pragma unroll
        for (int r = 0; r < 8; r++) park1[r * kThreads + t] = v[0][r];
    }
    u64 v[1][8];
    ks_intt_ksd_regs<2, false>(dg, rkd, k, v, smem, t);
    const u64 *pc = c3 + (op * 3 + k) * 2 * kN;
    u64 *po = out + (op * 2 + k) * 2 * kN;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        u64 o0, o1;
        ks_finish_coeff_ksd(park0[r * kThreads + t], park1[r * kThreads + t], v[0][r], pc[r * kThreads + t], pc[kN + r * kThreads + t], o0, o1);
        po[r * kThreads + t] = o0;
        po[kN + r * kThreads + t] = o1;
    }
}

// =====================================================================================
// K9b: rounded division by P and accumulation into (c0, c1)   (tail of switch_key_inplace)
//   out[op][k][l][i] = c3[op][k][l][i] + (ks[k][l][i] - ((ks[k][P][i] + P/2 mod P) mod q_l - (P/2 mod q_l))) * P^-1 mod q_l
// =====================================================================================
__global__ void __launch_bounds__(256) k_relin_finish(const u64 *__restrict__ c3, const u64 *__restrict__ ks,
                                                      u64 *__restrict__ out, size_t n_ops) {
    using Q0 = Mod<MQ0>;
    using Q1 = Mod<MQ1>;
    using PP = Mod<MP>;
    size_t total = n_ops * 2 * kN;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += stride) {
        size_t op = g / (2 * kN);
        int k = (int)((g / kN) & 1);
        int i = (int)(g % kN);
        const u64 *pk = ks + (op * 2 + k) * 3 * kN + i;
        const u64 *pc = c3 + (op * 3 + k) * 2 * kN + i;
        u64 *po = out + (op * 2 + k) * 2 * kN + i;
        u64 last = csub<PP>(pk[2 * kN] + kc.half_P, PP::q);
        {
            u64 tl = submod<Q0>(canon_k32<Q0>(last), kc.half_P_mod_q[0]);  // last < P < 4 q_l
            u64 d = submod<Q0>(pk[0], tl);
            po[0] = canon_k32<Q0>(shoup_acc<Q0, 2>(pc[0], d, kc.inv_P_mod_q[0].w, kc.inv_P_mod_q[0].ws));  // < 6 q_l
        }
        {
            u64 tl = submod<Q1>(canon_k32<Q1>(last), kc.half_P_mod_q[1]);  // last < P < 4 q_l
            u64 d = submod<Q1>(pk[kN], tl);
            po[kN] = canon_k32<Q1>(shoup_acc<Q1, 2>(pc[kN], d, kc.inv_P_mod_q[1].w, kc.inv_P_mod_q[1].ws));  // < 6 q_l
        }
    }
}

// =====================================================================================
// K11a: decryption   (SEAL Decryptor::bfv_decrypt, size-2 ciphertexts; fhe.rs:688-699)
//   k_decrypt_dot   : x_l = c0_l + INTT(NTT(c1_l) * s_l)            grid (2 limbs, ops) -> xbuf [op][2][N]
//   k_decrypt_round : m = round(t * CRT(x_0, x_1) / q) mod t        per coefficient     -> plain [op][N] u16
// SEAL rounds through the {t, gamma} base conversion; the exact rounding below gives the same plaintext
// whenever the noise budget is positive.
// =====================================================================================
template <int MI>
__device__ __forceinline__ void decrypt_dot_body(const u64 *__restrict__ ct, const u64 *__restrict__ sk, u64 *__restrict__ x,
                                                 u64 *smem, int t) {
    using M = Mod<MI>;
    u64 v[1][8], s[8], c0[8];
    load_natural(ct + (size_t)(1 * 2 + MI) * kN, v[0], t);
    ntt_forward<M, 1, true>(v, smem, kt.twf[MI], t);
    load_chunk8_ldg(sk + (size_t)MI * kN, s, t);
#pragma unroll
    for (int r = 0; r < 8; r++) v[0][r] = mulmod<M>(v[0][r], s[r]);
    ntt_inverse<M, 1>(v, smem, kt.twi[MI], t, kc.ninv[MI], kc.ninv_w[MI]);
    load_natural(ct + (size_t)(0 * 2 + MI) * kN, c0, t);
#pragma unroll
    for (int r = 0; r < 8; r++) v[0][r] = addmod<M>(v[0][r], c0[r]);
    store_natural(x + (size_t)MI * kN, v[0], t);
}
__global__ void __launch_bounds__(kThreads, 2) k_decrypt_dot(const u64 *__restrict__ ct, const u64 *__restrict__ sk,
                                                              u64 *__restrict__ xbuf) {
    extern __shared__ __align__(16) u64 smem[];
    const size_t op = blockIdx.y;
    if (blockIdx.x == 0)
        decrypt_dot_body<MQ0>(ct + op * 4 * kN, sk, xbuf + op * 2 * kN, smem, threadIdx.x);
    else
        decrypt_dot_body<MQ1>(ct + op * 4 * kN, sk, xbuf + op * 2 * kN, smem, threadIdx.x);
}
// exhausted[op] (optional) is set when the op's invariant noise budget is 0 -- SEAL Decryptor::invariant_noise_budget:
// bit_count(q) - bit_count(max_i |t x_i mod q|, centred) - 1 <= 0, i.e. the centred remainder of some coefficient reaches
// 2^70 -- which sunscreen's Runtime::decrypt turns into an error (-> FailedDecryption, fhe.rs:640-643, 692-696).
__global__ void __launch_bounds__(256) k_decrypt_round(const u64 *__restrict__ xbuf, unsigned short *__restrict__ plain,
                                                       size_t n_ops, int *__restrict__ exhausted) {
    using Q0 = Mod<MQ0>;
    using Q1 = Mod<MQ1>;
    size_t total = n_ops * kN;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    const u64 qlo = kc.q_lo, qhi = kc.q_hi;
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += stride) {
        size_t op = g / kN;
        int i = (int)(g % kN);
        u64 v0 = shoup<Q0>(xbuf[(op * 2 + 0) * kN + i], kc.crt_inv[0].w, kc.crt_inv[0].ws);
        u64 v1 = shoup<Q1>(xbuf[(op * 2 + 1) * kN + i], kc.crt_inv[1].w, kc.crt_inv[1].ws);
        // X = v0*q1 + v1*q0 mod q   (< 2q before the subtraction)
        u64 lo = 0, hi = 0;
        mac128(lo, hi, v0, Q1::q);
        mac128(lo, hi, v1, Q0::q);
        if (hi > qhi || (hi == qhi && lo >= qlo)) {
            u64 nl = lo - qlo;
            hi = hi - qhi - (lo < qlo);
            lo = nl;
        }
        // long division of t*X by q, t = 2^12: 12 shift-subtract steps
        u32 quo = 0;
#pragma unroll
        for (int b = 0; b < kLogT; b++) {
            hi = (hi << 1) | (lo >> 63);
            lo <<= 1;
            bool ge = hi > qhi || (hi == qhi && lo >= qlo);
            if (ge) {
                u64 nl = lo - qlo;
                hi = hi - qhi - (lo < qlo);
                lo = nl;
            }
            quo = (quo << 1) | (ge ? 1u : 0u);
        }
        // round to nearest (ties up): floor((tX + (q-1)/2) / q) = quo + [rem + (q-1)/2 >= q]
        u64 sl = lo + kc.qhalf_lo;
        u64 sh = hi + kc.qhalf_hi + (sl < lo);
        const bool up = sh > qhi || (sh == qhi && sl >= qlo);
        if (up) quo += 1;
        plain[g] = (unsigned short)(quo & (kT - 1));
        if (exhausted) {
            // centred remainder: rem if it rounds down, q - rem if it rounds up; bits 70.. of the 128-bit value
            const u64 nh = up ? qhi - hi - (qlo < lo) : hi;
            if (nh >> 6) exhausted[op] = 1;
        }
    }
}

// =====================================================================================
// K11b: deterministic public-key encryption, bit-exact with the reference (fhe.rs:594-657 -> sunscreen 0.8.1
//       `encrypt_deterministic` -> Sunscreen's SEAL 4.0 fork built with SEAL_USE_GAUSSIAN_NOISE).  Pinned by the reference's
//       SHA-512 known answers (tests/test_gpu_parity.py::test_reference_known_answers_through_the_c_abi).
//   k_seal_prng    : SEAL's Blake2xbPRNG stream for the op's 512-bit seed: buffer c (4096 bytes) = BLAKE2Xb(in = c as LE
//                    u64, key = seed).  The buffers and the 64 expansion nodes of a buffer are independent, so one CTA per
//                    op computes kSealBuffers roots and then 64 x kSealBuffers one-block BLAKE2b compressions in parallel.
//   k_seal_sample  : SEAL's samplers on that stream, in SEAL's order with one PRNG: sample_poly_ternary
//                    (std::uniform_int_distribution<uint64_t>(0, 2), libstdc++ >= 11 = Lemire on 32-bit draws), then
//                    sample_poly_normal twice (ClippedNormalDistribution(0, 3.2, 19.2) over libstdc++'s Marsaglia-polar
//                    std::normal_distribution<double>, truncated toward zero).  Draw consumption is data dependent
//                    (rejections), so acceptance flags are computed in parallel and compacted with a block scan; the rare
//                    cases (a zero draw in u, a clipped variate) take an exact sequential path on one thread.
//                    IEEE double arithmetic without contraction; log() is CUDA's (<= 1 ulp from glibc's), which can move
//                    a sample only if the scaled variate lies within ~2^-48 of an integer (~1e-11 per ciphertext).
//   k_encrypt_seal : encrypt_zero_asymmetric at the DATA level (the fork's deterministic encrypt disables the special
//                    modulus: the first two limbs of each public-key polynomial, no divide_and_round_q_last) +
//                    multiply_add_plain_with_scaling_variant:  c_j = INTT(NTT(u) * pk_j) + e_j,  c_0 += scaled(m).
//                    grid (2 limbs, ops) -> ct [op][2][2][N]
// =====================================================================================
constexpr int kSealBuffers = 28;                   // 28 x 4096 bytes = 28,672 draws; a ciphertext consumes ~25,000 (sigma ~150)
constexpr int kSealStreamWords = kSealBuffers * 512;  // u64 words of stream per op; the samples (3 x N int8) follow it
constexpr int kSealAttempts = 6;                   // polar attempts per thread and error polynomial (512 x 6 >= 2,608 +- 27)

#define B2B_G(a, b, c, d, x, y)                \
    a = a + b + (x), d = rotr64(d ^ a, 32);    \
    c = c + d, b = rotr64(b ^ c, 24);          \
    a = a + b + (y), d = rotr64(d ^ a, 16);    \
    c = c + d, b = rotr64(b ^ c, 63);
#define B2B_ROUND(s0, s1, s2, s3, s4, s5, s6, s7, s8, s9, s10, s11, s12, s13, s14, s15) \
    B2B_G(v[0], v[4], v[8], v[12], m[s0], m[s1])                                       \
    B2B_G(v[1], v[5], v[9], v[13], m[s2], m[s3])                                       \
    B2B_G(v[2], v[6], v[10], v[14], m[s4], m[s5])                                      \
    B2B_G(v[3], v[7], v[11], v[15], m[s6], m[s7])                                      \
    B2B_G(v[0], v[5], v[10], v[15], m[s8], m[s9])                                      \
    B2B_G(v[1], v[6], v[11], v[12], m[s10], m[s11])                                    \
    B2B_G(v[2], v[7], v[8], v[13], m[s12], m[s13])                                     \
    B2B_G(v[3], v[4], v[9], v[14], m[s14], m[s15])
__device__ __forceinline__ u64 rotr64(u64 x, int n) { return (x >> n) | (x << (64 - n)); }
__device__ __forceinline__ u64 b2b_iv(int i) {
    constexpr u64 iv[8] = {0x6A09E667F3BCC908ull, 0xBB67AE8584CAA73Bull, 0x3C6EF372FE94F82Bull, 0xA54FF53A5F1D36F1ull,
                           0x510E527FADE682D1ull, 0x9B05688C2B3E6C1Full, 0x1F83D9ABFB41BD6Bull, 0x5BE0CD19137E2179ull};
    return iv[i];
}
// BLAKE2b compression F (RFC 7693 3.2) with t < 2^64: h <- F(h, m, t, last)
__device__ __noinline__ void b2b_compress(u64 *__restrict__ h, const u64 *__restrict__ m_in, u64 t, bool last) {
    u64 v[16], m[16];
#pragma unroll
    for (int i = 0; i < 16; i++) m[i] = m_in[i];
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = h[i], v[i + 8] = b2b_iv(i);
    v[12] ^= t;
    if (last) v[14] = ~v[14];
    B2B_ROUND(0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15)
    B2B_ROUND(14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3)
    B2B_ROUND(11, 8, 12, 0, 5, 2, 15, 13, 10, 14, 3, 6, 7, 1, 9, 4)
    B2B_ROUND(7, 9, 3, 1, 13, 12, 11, 14, 2, 6, 5, 10, 4, 0, 15, 8)
    B2B_ROUND(9, 0, 5, 7, 2, 4, 10, 15, 14, 1, 11, 12, 6, 8, 3, 13)
    B2B_ROUND(2, 12, 6, 10, 0, 11, 8, 3, 4, 13, 7, 5, 15, 14, 1, 9)
    B2B_ROUND(12, 5, 1, 15, 14, 13, 4, 10, 0, 7, 6, 3, 9, 2, 8, 11)
    B2B_ROUND(13, 11, 7, 14, 12, 1, 3, 9, 5, 0, 15, 4, 8, 6, 2, 10)
    B2B_ROUND(6, 15, 14, 9, 11, 3, 0, 8, 12, 2, 13, 7, 1, 4, 10, 5)
    B2B_ROUND(10, 2, 8, 4, 7, 6, 1, 5, 15, 11, 9, 14, 3, 12, 13, 0)
    B2B_ROUND(0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15)
    B2B_ROUND(14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3)
#pragma unroll
    for (int i = 0; i < 8; i++) h[i] ^= v[i] ^ v[i + 8];
}
// h = IV xor parameter block (words 0..2 carry everything BLAKE2X sets; salt / personalisation are zero)
__device__ __forceinline__ void b2b_init(u64 *h, u64 digest, u64 keylen, u64 fanout, u64 depth, u64 leaf, u64 node_offset, u64 xof,
                                         u64 inner) {
#pragma unroll
    for (int i = 0; i < 8; i++) h[i] = b2b_iv(i);
    h[0] ^= digest | (keylen << 8) | (fanout << 16) | (depth << 24) | (leaf << 32);
    h[1] ^= node_offset | (xof << 32);
    h[2] ^= inner << 8;
}
__global__ void __launch_bounds__(512) k_seal_prng(const u64 *__restrict__ seeds, u64 *__restrict__ scratch, size_t op_stride) {
    __shared__ u64 roots[kSealBuffers][8];
    const size_t op = blockIdx.x;
    const u64 *seed = seeds + op * 8;
    u64 *stream = scratch + op * op_stride;
    const int t = threadIdx.x;
    if (t < kSealBuffers) {
        u64 h[8], m[16];
        b2b_init(h, 64, 64, 1, 1, 0, 0, 4096, 0);
#pragma unroll
        for (int i = 0; i < 16; i++) m[i] = i < 8 ? seed[i] : 0;  // the key, zero padded to one block
        b2b_compress(h, m, 128, false);
#pragma unroll
        for (int i = 0; i < 16; i++) m[i] = 0;
        m[0] = (u64)t;  // the buffer counter, 8 bytes of input
        b2b_compress(h, m, 136, true);
#pragma unroll
        for (int i = 0; i < 8; i++) roots[t][i] = h[i];
    }
    __syncthreads();
    for (int idx = t; idx < kSealBuffers * 64; idx += 512) {
        const int b = idx >> 6, node = idx & 63;
        u64 h[8], m[16];
        b2b_init(h, 64, 0, 0, 0, 64, (u64)node, 4096, 64);
#pragma unroll
        for (int i = 0; i < 16; i++) m[i] = i < 8 ? roots[b][i] : 0;
        b2b_compress(h, m, 64, true);
        uint4 *dst = reinterpret_cast<uint4 *>(stream + (size_t)b * 512 + node * 8);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            u32 a0, a1, a2, a3;
            unpack64(h[2 * i], a0, a1);
            unpack64(h[2 * i + 1], a2, a3);
            dst[i] = make_uint4(a0, a1, a2, a3);
        }
    }
}

// libstdc++ generate_canonical<double, 53> over a 32-bit engine: two draws, low word first
__device__ __forceinline__ double seal_canonical(u32 lo, u32 hi) {
    const double sum = __dadd_rn(__uint2double_rn(lo), __dmul_rn(__uint2double_rn(hi), 4294967296.0));
    const double r = __dmul_rn(sum, 5.42101086242752217e-20);  // / 2^64, exact
    return r >= 1.0 ? 0.99999999999999989 : r;                   // nextafter(1, 0)
}
// one Marsaglia-polar attempt on draws w[0..3]; returns acceptance
__device__ __forceinline__ bool seal_polar(const u32 *__restrict__ w, double &x, double &y, double &r2) {
    x = __dadd_rn(__dmul_rn(2.0, seal_canonical(w[0], w[1])), -1.0);
    y = __dadd_rn(__dmul_rn(2.0, seal_canonical(w[2], w[3])), -1.0);
    r2 = __dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y));
    return !(r2 > 1.0 || r2 == 0.0);
}
// the two variates of an accepted attempt, scaled by sigma, in the order std::normal_distribution returns them
__device__ __forceinline__ void seal_pair(double x, double y, double r2, double &first, double &second) {
    const double mult = __dsqrt_rn(__ddiv_rn(__dmul_rn(-2.0, log(r2)), r2));
    first = __dmul_rn(__dmul_rn(y, mult), 3.2);
    second = __dmul_rn(__dmul_rn(x, mult), 3.2);
}
// exact sequential sample_poly_normal from draw index `base` (one thread): returns draws consumed, 0 if the stream ran out
__device__ __noinline__ u32 seal_normal_sequential(const u32 *__restrict__ w, u32 base, u32 limit, signed char *__restrict__ out) {
    u32 pos = base;
    bool have = false;
    double saved = 0.0;
    for (int i = 0; i < kN; i++) {
        double value;
        for (;;) {
            if (have) {
                have = false, value = saved;
            } else {
                double x, y, r2;
                for (;;) {
                    if (pos + 4 > limit) return 0;
                    const bool ok = seal_polar(w + pos, x, y, r2);
                    pos += 4;
                    if (ok) break;
                }
                seal_pair(x, y, r2, value, saved);
                have = true;
            }
            if (fabs(value) <= 19.2) break;
        }
        out[i] = (signed char)__double2int_rz(value);
    }
    return pos - base;
}
// exclusive prefix sum of `v` over the 512 threads of the block; *total = sum
__device__ __forceinline__ int block_exclusive_scan(int v, int *warp_sums, int *total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int n = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += n;
    }
    if (lane == 31) warp_sums[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        int s = lane < 16 ? warp_sums[lane] : 0;
#pragma unroll
        for (int d = 1; d < 16; d <<= 1) {
            int n = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += n;
        }
        if (lane < 16) warp_sums[16 + lane] = s;  // inclusive sums of the warps
    }
    __syncthreads();
    *total = warp_sums[31];
    const int before = wid ? warp_sums[16 + wid - 1] : 0;
    __syncthreads();
    return before + inc - v;
}
__global__ void __launch_bounds__(512) k_seal_sample(u64 *__restrict__ scratch, size_t op_stride, int *__restrict__ failed) {
    __shared__ int warp_sums[32];
    __shared__ u32 sh_consumed;
    __shared__ int sh_slow;
    const size_t op = blockIdx.x;
    const u32 *w = reinterpret_cast<const u32 *>(scratch + op * op_stride);
    signed char *smp = reinterpret_cast<signed char *>(scratch + op * op_stride + kSealStreamWords);
    const u32 limit = (u32)kSealStreamWords * 2;
    const int t = threadIdx.x;
    // ---- u: draw i gives floor(3 w / 2^32) unless w == 0 (Lemire: low word 0 < threshold 1 -> redraw)
    int zeros = 0;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const u32 x = w[r * 512 + t];
        zeros += x == 0;
        smp[r * 512 + t] = (signed char)((int)__umulhi(x, 3u) - 1);
    }
    zeros = __syncthreads_count(zeros);
    u32 base = kN;
    if (zeros) {  // ~1e-6 of the seeds: the exact walk on one thread
        if (t == 0) {
            u32 pos = 0;
            for (int i = 0; i < kN; i++) {
                u32 x;
                do x = w[pos++];
                while (x == 0);
                smp[i] = (signed char)((int)__umulhi(x, 3u) - 1);
            }
            sh_consumed = pos;
        }
        __syncthreads();
        base = sh_consumed;
        __syncthreads();
    }
    // ---- e0, e1
    bool ok = true;
    for (int j = 0; j < 2; j++) {
        signed char *e = smp + (1 + j) * kN;
        if (t == 0) sh_slow = 0, sh_consumed = 0;
        int acc = 0;
#pragma unroll
        for (int r = 0; r < kSealAttempts; r++) {
            const u32 idx = base + 4u * (u32)(t * kSealAttempts + r);
            double x, y, r2;
            if (idx + 4 <= limit) acc += seal_polar(w + idx, x, y, r2) ? 1 : 0;
        }
        int total;
        int p = block_exclusive_scan(acc, warp_sums, &total);  // syncs; sh_slow / sh_consumed are initialised past here
#pragma unroll
        for (int r = 0; r < kSealAttempts; r++) {
            const u32 k = (u32)(t * kSealAttempts + r);
            const u32 idx = base + 4u * k;
            double x, y, r2;
            if (idx + 4 <= limit && seal_polar(w + idx, x, y, r2)) {
                if (p < kN / 2) {
                    double a, b;
                    seal_pair(x, y, r2, a, b);
                    if (fabs(a) > 19.2 || fabs(b) > 19.2) sh_slow = 1;  // a clipped variate shifts everything behind it
                    e[2 * p] = (signed char)__double2int_rz(a);
                    e[2 * p + 1] = (signed char)__double2int_rz(b);
                    if (p == kN / 2 - 1) sh_consumed = 4u * (k + 1);
                }
                p++;
            }
        }
        __syncthreads();
        if (sh_slow || total < kN / 2) {  // exact sequential path (also when the window of attempts was too short)
            if (t == 0) sh_consumed = seal_normal_sequential(w, base, limit, e);
            __syncthreads();
        }
        const u32 used = sh_consumed;
        __syncthreads();
        if (!used) ok = false;
        base += used;
    }
    if (t == 0 && failed) failed[op] = ok ? 0 : 1;
}
template <int MI>
__device__ __forceinline__ void encrypt_seal_body(const u64 *__restrict__ pk, const signed char *__restrict__ smp,
                                                  const unsigned short *__restrict__ plain, u64 *__restrict__ ct, u64 *smem, int t) {
    using M = Mod<MI>;
    u64 v[1][8];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const int u = smp[r * kThreads + t];
        v[0][r] = u < 0 ? M::q - 1 : (u64)u;
    }
    ntt_forward<M, 1, true>(v, smem, kt.twf[MI], t);
    u64 w[2][8];
#pragma unroll
    for (int j = 0; j < 2; j++) {
        u64 k[8];
        load_chunk8_ldg(pk + (size_t)(j * 3 + MI) * kN, k, t);
#pragma unroll
        for (int r = 0; r < 8; r++) w[j][r] = mulmod<M>(v[0][r], k[r]);
    }
    ntt_inverse<M, 2>(w, smem, kt.twi[MI], t, kc.ninv[MI], kc.ninv_w[MI]);
#pragma unroll
    for (int j = 0; j < 2; j++) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const int e = smp[(1 + j) * kN + r * kThreads + t];
            const u64 ev = e < 0 ? M::q - (u64)(-e) : (u64)e;
            u64 x = addmod<M>(w[j][r], ev);
            if (j == 0) x = addmod<M>(x, plain_scaled<M>(plain[r * kThreads + t], MI));
            w[j][r] = x;
        }
        store_natural(ct + (size_t)(j * 2 + MI) * kN, w[j], t);
    }
}
// pks [k][2][3][N]: op i encrypts under pks + key_index[i] * 6N, or under pks itself when key_index is null
__global__ void __launch_bounds__(kThreads, 1) k_encrypt_seal(const u64 *__restrict__ pks, const int *__restrict__ key_index,
                                                               const u64 *__restrict__ scratch, size_t op_stride,
                                                               const unsigned short *__restrict__ plain, u64 *__restrict__ ct) {
    extern __shared__ __align__(16) u64 smem[];
    const size_t op = blockIdx.y;
    const u64 *pk = pks + (key_index ? (size_t)key_index[op] : 0) * (6 * kN);
    const signed char *smp = reinterpret_cast<const signed char *>(scratch + op * op_stride + kSealStreamWords);
    const unsigned short *pl = plain + op * kN;
    u64 *out = ct + op * 4 * kN;
    if (blockIdx.x == 0)
        encrypt_seal_body<MQ0>(pk, smp, pl, out, smem, threadIdx.x);
    else
        encrypt_seal_body<MQ1>(pk, smp, pl, out, smem, threadIdx.x);
}

// =====================================================================================
// integer-pipe peak microbenchmark (roofline denominator for the multiply kernels; not on the hot path)
// 16 independent mad chains per thread; WIDE: mad.wide.u32 (32x32+64 -> 64), else mad.lo.u32
// =====================================================================================
// MODE 0: mad.lo.u32 (IMAD), 1: mul.wide.u32 (IMAD.WIDE), 2: add.cc/addc pairs (IADD3 + IADD3.X, counted as 2 ops),
//      3: mad.lo + add interleaved (counts both), 4: mul.wide + add interleaved (counts both).
// Every multiply has a loop-carried multiplicand so that ptxas cannot strength-reduce it.
template <int MODE>
__global__ void __launch_bounds__(1024) k_int_peak(u64 *out, int iters, u32 a, u32 b) {
    u32 x[16], y[16];
#pragma unroll
    for (int j = 0; j < 16; j++) {
        x[j] = threadIdx.x * 77u + j + a;
        y[j] = threadIdx.x * 13u + j * b;
    }
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int j = 0; j < 16; j++) {
            if (MODE == 0 || MODE == 3) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[j]) : "r"(a), "r"(b));
            if (MODE == 1 || MODE == 4) {
                u64 t;
                asm volatile("mul.wide.u32 %0, %1, %2;" : "=l"(t) : "r"(x[j]), "r"(a));
                x[j] = (u32)(t >> 32) + (u32)t;  // one extra add keeps both halves live
            }
            if (MODE == 2) asm volatile("add.cc.u32 %0, %0, %2;\n\taddc.u32 %1, %1, %3;" : "+r"(x[j]), "+r"(y[j]) : "r"(a), "r"(b));
            if (MODE == 3 || MODE == 4) asm volatile("add.u32 %0, %0, %1;" : "+r"(y[j]) : "r"(a));
        }
    }
    u32 r = 0;
#pragma unroll
    for (int j = 0; j < 16; j++) r ^= x[j] ^ y[j];
    if (r == 0x12345u) out[0] = r;
}

// Register-only butterfly throughput: every thread runs `iters` forward radix-8 passes (12 butterflies each)
// on 8 resident values with twiddles held in registers -- the practical integer-pipe ceiling of the NTT inner
// loop, free of memory and barrier effects.
template <int MI, int NV, int THREADS>
__global__ void __launch_bounds__(THREADS) k_bfly_peak(u64 *out, int iters, ulonglong2 tw0) {
    using M = Mod<MI>;
    u64 v[NV];
#pragma unroll
    for (int r = 0; r < NV; r++) v[r] = ((threadIdx.x * NV + r) * 0x9E3779B97F4A7C15ull >> 8) % M::q;
    u64 w = tw0.x % M::q, ws = tw0.y;
    for (int i = 0; i < iters; i++) {
        // log2(NV) butterfly stages over the NV resident values (stage indices chosen so that the 61-bit path folds
        // once every third stage, as in the real transform)
#pragma unroll
        for (int r = 0; r < NV / 2; r++) fwd_bfly<M, 3>(v[r], v[r + NV / 2], w, ws);
#pragma unroll
        for (int r = 0; r < NV / 2; r++) fwd_bfly<M, 4>(v[(r / (NV / 4)) * (NV / 2) + r % (NV / 4)], v[(r / (NV / 4)) * (NV / 2) + r % (NV / 4) + NV / 4], w, ws);
#pragma unroll
        for (int r = 0; r < NV / 2; r++) fwd_bfly<M, 5>(v[2 * r], v[2 * r + 1], w, ws);
        if (M::kSmall) {  // keep the lazy values inside the range the real transform guarantees
#pragma unroll
            for (int r = 0; r < NV; r++) v[r] &= (1ull << 40) - 1;
        }
    }
    u64 acc = 0;
#pragma unroll
    for (int r = 0; r < NV; r++) acc ^= v[r];
    if (acc == tw0.x) out[0] = acc;
}
template <int MI, int NV, int THREADS>
static float time_bfly(u64 *d, int iters, int grid, ulonglong2 tw) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        cudaEventRecord(e0);
        k_bfly_peak<MI, NV, THREADS><<<grid, THREADS>>>(d, iters, tw);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return best;
}
// mod 0-2: small primes, 3-5: 61-bit; mod + 10: 16 values per thread / 256 threads (ILP experiment)
cudaError_t measure_bfly_peak(int mod, double *giga_bfly_per_s) {
    u64 *d = nullptr;
    cudaError_t e = cudaMalloc((void **)&d, 8);
    if (e != cudaSuccess) return e;
    const int iters = 2048;
    ulonglong2 tw = make_ulonglong2(0x123456789ull, 0x9abcdef012345678ull);
    float ms;
    double bfly;
    if (mod >= 10) {
        const int grid = 148 * 8;
        ms = (mod - 10) < 3 ? time_bfly<MQ0, 16, 256>(d, iters, grid, tw) : time_bfly<MB0, 16, 256>(d, iters, grid, tw);
        bfly = (double)grid * 256 * iters * 24.0;
    } else {
        const int grid = 148 * 4;
        ms = mod < 3 ? time_bfly<MQ0, 8, kThreads>(d, iters, grid, tw) : time_bfly<MB0, 8, kThreads>(d, iters, grid, tw);
        bfly = (double)grid * kThreads * iters * 12.0;
    }
    cudaFree(d);
    *giga_bfly_per_s = bfly / (ms * 1e-3) / 1e9;
    return cudaGetLastError();
}

// result: 1e12 thread-level operations per second (see the MODE list above for what is counted)
cudaError_t measure_int_peak(int mode, double *tera_ops_per_s) {
    u64 *d = nullptr;
    cudaError_t e = cudaMalloc((void **)&d, 8);
    if (e != cudaSuccess) return e;
    const int iters = 4096, grid = 148 * 2, block = 1024;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        cudaEventRecord(e0);
        switch (mode) {
            case 0: k_int_peak<0><<<grid, block>>>(d, iters, 3, 5); break;
            case 1: k_int_peak<1><<<grid, block>>>(d, iters, 3, 5); break;
            case 2: k_int_peak<2><<<grid, block>>>(d, iters, 3, 5); break;
            case 3: k_int_peak<3><<<grid, block>>>(d, iters, 3, 5); break;
            default: k_int_peak<4><<<grid, block>>>(d, iters, 3, 5); break;
        }
        cudaEventRecord(e1);
        e = cudaEventSynchronize(e1);
        if (e != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    if (e != cudaSuccess) return e;
    const double per = (mode == 2 || mode == 3 || mode == 4) ? 2.0 : 1.0;
    *tera_ops_per_s = (double)grid * block * iters * 16.0 * per / (best * 1e-3) / 1e12;
    return cudaGetLastError();
}

// =====================================================================================
// launchers
// =====================================================================================
static const int kSmem1 = 1 * kN * 8, kSmem2 = 2 * kN * 8, kSmem3 = 3 * kN * 8;

cudaError_t kernels_configure() {
    cudaError_t e;
    e = cudaFuncSetAttribute(k_mul_plain, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem3);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_encrypt_seal, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem2);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_tensor_floor_d, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem3);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_ks_tail_ksd, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem3);
    if (e != cudaSuccess) return e;
    return cudaSuccess;
}

static std::atomic<unsigned long long> g_launches{0};
uint64_t launch_count() { return g_launches.load(); }
void count_launches(uint64_t n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

static int eltwise_grid(size_t n, int block) {
    size_t g = (n + block - 1) / block;
    size_t cap = 148 * 16;
    return (int)(g < cap ? (g ? g : 1) : cap);
}

cudaError_t launch_ntt(u64 *data, size_t n_limbs, const LimbMods &mods, bool inverse, cudaStream_t s) {
    if (n_limbs == 0) return cudaSuccess;
    if (inverse) k_ntt<true><<<(unsigned)n_limbs, kThreads, kSmem1, s>>>(data, mods);
    else k_ntt<false><<<(unsigned)n_limbs, kThreads, kSmem1, s>>>(data, mods);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

cudaError_t launch_eltwise(const u64 *a, const u64 *b, u64 *out, size_t n_ops, int op, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    size_t n2 = n_ops * 4 * kN / 2;
    k_eltwise<<<eltwise_grid(n2, 256), 256, 0, s>>>((const ulonglong2 *)a, (const ulonglong2 *)b, (ulonglong2 *)out, n2, op);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

cudaError_t launch_plain_addsub(const u64 *ct, const unsigned short *plain, u64 *out, size_t n_ops, int mode, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    k_plain_addsub<<<eltwise_grid(n_ops * 4 * kN, 256), 256, 0, s>>>(ct, plain, out, n_ops, mode);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

cudaError_t launch_mul_plain(const u64 *ct, const unsigned short *plain, u64 *out, size_t n_ops, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    for (size_t done = 0; done < n_ops;) {
        size_t c = n_ops - done < 65535 ? n_ops - done : 65535;
        k_mul_plain<<<dim3(2, (unsigned)c), kThreads, kSmem3, s>>>(ct + done * 4 * kN, plain + done * kN, out + done * 4 * kN);
        if (done) g_launches.fetch_add(1, std::memory_order_relaxed);
        done += c;
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

cudaError_t launch_ext_conv(const u64 *a, const u64 *b, u64 *nttbuf, size_t n_ops, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    k_ext_conv_d<<<eltwise_grid(n_ops * 4 * (kN / 2), 256), 256, 0, s>>>(a, b, nttbuf, n_ops);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_ext_ntt(u64 *nttbuf, size_t n_ops, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    k_ext_ntt_d<<<dim3(12, (unsigned)n_ops), kThreads, kSmem1, s>>>(nttbuf);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_tensor_intt(const u64 *nttbuf, u64 *tens, size_t n_ops, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    k_tensor_intt_d<<<dim3(9, (unsigned)n_ops), kThreads, kSmem1, s>>>(nttbuf, tens);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_floor_sk(const u64 *tens, u64 *c3, size_t n_ops, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    k_floor_sk_d<<<eltwise_grid(n_ops * 3 * (kN / 2), 256), 256, 0, s>>>(tens, c3, n_ops);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_tensor_floor(const u64 *nttbuf, u64 *c3, size_t n_ops, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    k_tensor_floor_d<<<dim3(3, (unsigned)n_ops), kThreads, kSmem3, s>>>(nttbuf, c3);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_ks_tail_ksd(const u64 *dig, const u64 *rkd, const u64 *c3, u64 *out, size_t n_ops, cudaStream_t s,
                               const int *key_index) {
    if (n_ops == 0) return cudaSuccess;
    k_ks_tail_ksd<<<dim3(2, (unsigned)n_ops), kThreads, kSmem3, s>>>(dig, rkd, key_index, c3, out);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_digit_ntt(const u64 *c3, u64 *dig, size_t n_ops, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    k_digit_ntt<<<dim3(6, (unsigned)n_ops), kThreads, kSmem1, s>>>(c3, dig);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_ks_intt(const u64 *dig, const u64 *rk, u64 *ks, size_t n_ops, cudaStream_t s) {
    return launch_ks_intt_keyed(dig, rk, nullptr, nullptr, ks, n_ops, s);
}
cudaError_t launch_ks_intt_keyed(const u64 *dig, const u64 *rk, const u64 *const *rks, const int *key_index, u64 *ks, size_t n_ops,
                                 cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    k_ks_intt<<<dim3(6, (unsigned)n_ops), kThreads, kSmem1, s>>>(dig, rk, rks, key_index, ks);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_decrypt(const u64 *ct, const u64 *sk, u64 *xbuf, unsigned short *plain, size_t n_ops, cudaStream_t s,
                           int *exhausted) {
    if (n_ops == 0) return cudaSuccess;
    if (exhausted) {
        cudaError_t e = cudaMemsetAsync(exhausted, 0, n_ops * sizeof(int), s);
        if (e != cudaSuccess) return e;
    }
    k_decrypt_dot<<<dim3(2, (unsigned)n_ops), kThreads, kSmem1, s>>>(ct, sk, xbuf);
    k_decrypt_round<<<eltwise_grid(n_ops * kN, 256), 256, 0, s>>>(xbuf, plain, n_ops, exhausted);
    g_launches.fetch_add(2, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_encrypt_keyed(const u64 *pks, const int *key_index, const unsigned short *plain, const u64 *seeds, u64 *encbuf,
                                 u64 *ct, size_t n_ops, cudaStream_t s, int *failed) {
    if (n_ops == 0) return cudaSuccess;
    static_assert(kSealStreamWords + 3 * kN / 8 <= 6 * kN, "per-op encryption scratch is [6][N] words");
    const size_t stride = 6 * kN;
    k_seal_prng<<<(unsigned)n_ops, 512, 0, s>>>(seeds, encbuf, stride);
    k_seal_sample<<<(unsigned)n_ops, 512, 0, s>>>(encbuf, stride, failed);
    k_encrypt_seal<<<dim3(2, (unsigned)n_ops), kThreads, kSmem2, s>>>(pks, key_index, encbuf, stride, plain, ct);
    g_launches.fetch_add(3, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_encrypt(const u64 *pk, const unsigned short *plain, const u64 *seeds, u64 *encbuf, u64 *ct, size_t n_ops,
                           cudaStream_t s, int *failed) {
    return launch_encrypt_keyed(pk, nullptr, plain, seeds, encbuf, ct, n_ops, s, failed);
}
cudaError_t launch_seal_sample(u64 *streams, signed char *samples, int *failed, size_t n_ops, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    const size_t stride = (size_t)kSealStreamWords + 3 * kN / 8;
    k_seal_sample<<<(unsigned)n_ops, 512, 0, s>>>(streams, stride, failed);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    (void)samples;  // the samples are written behind each op's stream words (see kernels.h)
    return cudaGetLastError();
}
// the key of the key switch on the dual base, once per chunk; tmp = 36 limbs of scratch (coefficient-form key, lifted key,
// dual-NTT key at tmp + 24 limbs)
cudaError_t launch_rk_prepare_ksd(const u64 *rk, u64 *tmp, cudaStream_t s) {
    return launch_rk_prepare_keys(rk, nullptr, 1, tmp, tmp + 24 * kN, s);
}
cudaError_t launch_rk_prepare_keys(const u64 *rk, const u64 *const *rks, size_t n_keys, u64 *tmp, u64 *rkd, cudaStream_t s) {
    if (n_keys == 0) return cudaSuccess;
    if (n_keys > kMaxPrepareKeys) return cudaErrorInvalidValue;
    u64 *coef = tmp, *lifted = tmp + n_keys * 12 * kN;
    k_rk_intt_ksd<<<dim3(12, (unsigned)n_keys), kThreads, kSmem1, s>>>(rk, rks, coef);
    k_rk_lift_ksd<<<(unsigned)(n_keys * 4 * kN / 256), 256, 0, s>>>(coef, lifted);
    k_rk_ntt_ksd<<<(unsigned)(n_keys * 12), kThreads, kSmem1, s>>>(lifted, rkd);
    g_launches.fetch_add(3, std::memory_order_relaxed);
    return cudaGetLastError();
}
__global__ void k_key_table(const u64 *rks, size_t stride, size_t n_keys, const u64 **table) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_keys) table[i] = rks + i * stride;
}
cudaError_t launch_key_table(const u64 *rks, size_t stride, size_t n_keys, const u64 **table, cudaStream_t s) {
    if (n_keys == 0) return cudaSuccess;
    k_key_table<<<(unsigned)((n_keys + 255) / 256), 256, 0, s>>>(rks, stride, n_keys, table);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_digit_ntt_ksd(const u64 *c3, u64 *dig, size_t n_ops, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    k_digit_ntt_ksd<<<dim3(6, (unsigned)n_ops), kThreads, kSmem1, s>>>(c3, dig);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}
cudaError_t launch_relin_finish(const u64 *c3, const u64 *ks, u64 *out, size_t n_ops, cudaStream_t s) {
    if (n_ops == 0) return cudaSuccess;
    k_relin_finish<<<eltwise_grid(n_ops * 2 * kN, 256), 256, 0, s>>>(c3, ks, out, n_ops);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

}  // namespace fheb
