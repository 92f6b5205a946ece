// Negacyclic NTT building blocks, N = 4096, one CTA of 512 threads, 8 coefficients per thread.
// Replaces SEAL ntt_negacyclic_harvey / inverse_ntt_negacyclic_harvey (util/ntt.h, dwthandler.h)
// as used by Evaluator::bfv_multiply / switch_key_inplace / multiply_plain on the reference's hot
// path (FheApp::run, /root/reference/src/fhe.rs:138-152).  Same transform: forward takes natural
// order to bit-reversed order with twiddle table rp[bitrev(i)] = psi^i, inverse undoes it and
// scales by a caller-supplied constant (N^-1, possibly merged with another scalar).
//
// Structure: the 12 radix-2 stages are grouped into 4 register-resident radix-8 passes.
// Pass with first stage S0 keeps index bits (11-S0, 10-S0, 9-S0) in registers; the other nine bits
// are the thread id.  Between passes the 8 values go through shared memory with an XOR swizzle that
// makes every pass's 64-bit accesses bank-conflict-free for a half warp (see swz()).
// Twiddles are (w, floor(w*2^64/q)) pairs read through the read-only path from an L2-resident table.
#pragma once
#include "devconsts.h"
#include "modarith.cuh"

namespace fheb {

constexpr int kThreads = 512;

// physical slot of logical coefficient i inside a 4096-entry shared buffer
__device__ __forceinline__ int swz(int i) { return i ^ ((i >> 4) & 7) ^ (((i >> 6) & 1) << 3); }

// The exchange between the first two passes involves the whole CTA; the one between passes S0=3 and S0=6 stays inside
// 64 consecutive threads (same index bits 11..9) and the one between S0=6 and S0=9 inside 8 consecutive threads (one
// warp), so they use a 2-warp named barrier and __syncwarp(): warps of one CTA drift apart and their memory phases
// overlap other warps' multiply phases.
__device__ __forceinline__ void sync_group64(int t) { asm volatile("bar.sync %0, 64;" ::"r"(1 + (t >> 6)) : "memory"); }

// logical index of register r (0..7) of thread t in the pass whose first stage is S0
template <int S0>
__device__ __forceinline__ int elem_index(int t, int r) {
    constexpr int LB = 9 - S0;
    int lower = t & ((1 << LB) - 1);
    int upper = t >> LB;
    return (upper << (12 - S0)) | (r << LB) | lower;
}

template <int S0>
__device__ __forceinline__ int pass_upper(int t) {
    return t >> (9 - S0);
}

// ---------------------------------------------------------------- butterflies
// forward (Cooley-Tukey): (X, Y) -> (X + wY, X - wY), lazily.  G = global stage index 0..11.
//  small primes: T = wY in [0,5q) (approximate Shoup quotient); bounds grow by 5q per stage, never reduced: inputs < 2^42 stay
//                 below 2^42 + 60q < 2^44 (< 2^43 from canonical inputs), inside shoup_acc<M, 2>'s x < 2^44.
//  61-bit primes: T in [0,2q); stage inputs grow 2q -> 4q -> 6q -> 8q (< 2^64) and X is folded back below 2q
//                 (3 instructions: q = 2^61 - c) on every third stage.
template <class M, int G>
__device__ __forceinline__ void fwd_bfly(u64 &X, u64 &Y, u64 w, u64 ws) {
    if constexpr (M::kDual) {
        dual_fwd_bfly<M>(X, Y, w, ws);
    } else if constexpr (M::kSmall) {
        const u64 Xo = shoup_acc<M, 2>(X, Y, w, ws);  // Y < 2^42 + 55q < 2^44 throughout the forward transform
        Y = (X + X + 5 * M::q) - Xo;  // X + 5q - T
        X = Xo;
    } else {
        u64 x = X;
        if (G > 0 && (G % 3) == 0) x = fold_k32<M>(x);  // < 8q  ->  < 2^61 + 7c < 2q
        const u64 Xo = shoup_acc<M, 0>(x, Y, w, ws);
        Y = (x + x + M::two_q) - Xo;  // x + 2q - T
        X = Xo;
    }
}
// inverse (Gentleman-Sande): (X, Y) -> (X + Y, w(X - Y)); G = global stage index 0..11
//  small primes: inputs < 4q * 2^G, X output < 4q * 2^(G+1), Y output < 4q; never reduced (< 2^51 at the end).
//  61-bit primes: even stages take inputs < 2q and leave X + Y < 4q unreduced; odd stages take inputs < 4q and
//                 fold X + Y (< 8q) back below 2q.  Y outputs are always < 2q.
template <class M, int G>
__device__ __forceinline__ void inv_bfly(u64 &X, u64 &Y, u64 w, u64 ws) {
    if constexpr (M::kDual) {
        dual_inv_bfly<M>(X, Y, w, ws);
    } else if constexpr (M::kSmall) {
        constexpr u64 K = M::four_q << G;
        const u64 D = X + (K - Y);
        X = X + Y;
        Y = shoup_acc<M, 1>(0, D, w, ws);  // D can reach 2^51: the 16-bit estimate of variant 2 does not apply
    } else if constexpr ((G % 2) == 0) {
        const u64 D = X + (M::two_q - Y);
        X = X + Y;
        Y = shoup_lazy<M>(D, w, ws);
    } else {
        const u64 D = X + (M::four_q - Y);
        X = fold_k32<M>(X + Y);
        Y = shoup_lazy<M>(D, w, ws);
    }
}

// twiddle (w, Shoup quotient) number i of modulus M: stages 0..5 (i < 64) come from constant memory (CTA- or
// warp-uniform addresses), the rest from the L2/L1-resident table through the read-only path
template <class M, bool kInv, int S0>
__device__ __forceinline__ ulonglong2 ldtw(const ulonglong2 *__restrict__ tw, int i) {
    if (S0 <= 3) return kInv ? ktl.i[M::kIndex][i] : ktl.f[M::kIndex][i];
    if (S0 == 9) {
        // the pass that owns stages 9..11: the slot-major copy behind the table (params.h kTwPass9), coalesced per warp.
        // i = 512 + t, 1024 + 2t + h or 2048 + 4t + h with h a compile-time constant after unrolling
        const int lvl = i >= 2048 ? 2 : (i >= 1024 ? 1 : 0);
        const int t = (i - (512 << lvl)) >> lvl, h = i & ((1 << lvl) - 1);
        return __ldg(tw + kN + ((1 << lvl) - 1 + h) * 512 + t);
    }
    return __ldg(tw + i);
}

// ---------------------------------------------------------------- register radix-8 passes
// v[p][r]: r = 4*r2 + 2*r1 + r0, r2 <-> index bit 11-S0 (largest gap)
template <class M, int NP, int S0>
__device__ __forceinline__ void fwd_pass(u64 (&v)[NP][8], const ulonglong2 *__restrict__ tw, int upper) {
    {
        ulonglong2 w = ldtw<M, false, S0>(tw, (1 << S0) + upper);
#pragma unroll
        for (int p = 0; p < NP; p++)
#pragma unroll
            for (int r = 0; r < 4; r++) fwd_bfly<M, S0>(v[p][r], v[p][r + 4], w.x, w.y);
    }
#pragma unroll
    for (int h = 0; h < 2; h++) {
        ulonglong2 w = ldtw<M, false, S0>(tw, (2 << S0) + 2 * upper + h);
#pragma unroll
        for (int p = 0; p < NP; p++)
#pragma unroll
            for (int r = 0; r < 2; r++) fwd_bfly<M, S0 + 1>(v[p][4 * h + r], v[p][4 * h + r + 2], w.x, w.y);
    }
#pragma unroll
    for (int h = 0; h < 4; h++) {
        ulonglong2 w = ldtw<M, false, S0>(tw, (4 << S0) + 4 * upper + h);
#pragma unroll
        for (int p = 0; p < NP; p++) fwd_bfly<M, S0 + 2>(v[p][2 * h], v[p][2 * h + 1], w.x, w.y);
    }
}

// last Gentleman-Sande stage (G = 11) with the output scaling merged in: (X, Y) -> (s(X + Y), s w (X - Y)),
// both through exact Shoup multiplications, results in [0, 2q) or canonical
template <class M, bool kCanon>
__device__ __forceinline__ void inv_bfly_last(u64 &X, u64 &Y, const Shoup &s, const Shoup &sw) {
    if constexpr (M::kDual) {
        dual_inv_bfly_last<M, kCanon>(X, Y, s.w, s.ws, sw.w, sw.ws);
        return;
    } else {
    constexpr u64 K = M::kSmall ? (M::four_q << 11) : M::four_q;  // >= the stage's input bound (odd stage: < 4q for 61-bit)
    const u64 D = X + (K - Y);
    const u64 S = X + Y;
    X = kCanon ? shoup<M>(S, s.w, s.ws) : shoup_lazy<M>(S, s.w, s.ws);
    Y = kCanon ? shoup<M>(D, sw.w, sw.ws) : shoup_lazy<M>(D, sw.w, sw.ws);
    }
}

// inverse pass over the same register bits, stages in reverse order. G0 = global index of its first stage.
// kLast (only with S0 == 0): the pass's final stage is the transform's last one and applies the scaling (s, sw).
template <class M, int NP, int S0, int G0, bool kLast = false, bool kCanon = true>
__device__ __forceinline__ void inv_pass(u64 (&v)[NP][8], const ulonglong2 *__restrict__ tw, int upper, const Shoup *s = nullptr,
                                         const Shoup *sw = nullptr) {
#pragma unroll
    for (int h = 0; h < 4; h++) {
        ulonglong2 w = ldtw<M, true, S0>(tw, (4 << S0) + 4 * upper + h);
#pragma unroll
        for (int p = 0; p < NP; p++) inv_bfly<M, G0>(v[p][2 * h], v[p][2 * h + 1], w.x, w.y);
    }
#pragma unroll
    for (int h = 0; h < 2; h++) {
        ulonglong2 w = ldtw<M, true, S0>(tw, (2 << S0) + 2 * upper + h);
#pragma unroll
        for (int p = 0; p < NP; p++)
#pragma unroll
            for (int r = 0; r < 2; r++) inv_bfly<M, G0 + 1>(v[p][4 * h + r], v[p][4 * h + r + 2], w.x, w.y);
    }
    if (kLast) {
#pragma unroll
        for (int p = 0; p < NP; p++)
#pragma unroll
            for (int r = 0; r < 4; r++) inv_bfly_last<M, kCanon>(v[p][r], v[p][r + 4], *s, *sw);
    } else {
        ulonglong2 w = ldtw<M, true, S0>(tw, (1 << S0) + upper);
#pragma unroll
        for (int p = 0; p < NP; p++)
#pragma unroll
            for (int r = 0; r < 4; r++) inv_bfly<M, G0 + 2>(v[p][r], v[p][r + 4], w.x, w.y);
    }
}

// ---------------------------------------------------------------- shared-memory exchange
// swz() is linear over GF(2) and only rewrites index bits 0..3, so the slot of register r is
//   swz(idx0 ^ (r << LB)) = swz(idx0) ^ swz(r << LB) = (base ^ X_r) + A_r
// with compile-time X_r (the part inside bits 0..3) and A_r (the rest, carry-free because idx0 is zero there).
// One base per pass, at most one LOP3 per access, the rest folds into the LDS/STS immediate offset.
__host__ __device__ constexpr int swz_c(int i) { return i ^ ((i >> 4) & 7) ^ (((i >> 6) & 1) << 3); }
template <int S0>
struct PassSlot {
    static constexpr int LB = 9 - S0;
    __host__ __device__ static constexpr int x(int r) { return swz_c(r << LB) & 0xF; }
    __host__ __device__ static constexpr int a(int r) { return swz_c(r << LB) & ~0xF; }
};
// smem: NP consecutive 4096-entry buffers
template <int NP, int S0>
__device__ __forceinline__ void smem_store(u64 *smem, const u64 (&v)[NP][8], int t) {
    const int base = swz(elem_index<S0>(t, 0));
#pragma unroll
    for (int p = 0; p < NP; p++)
#pragma unroll
        for (int r = 0; r < 8; r++) smem[p * kN + (base ^ PassSlot<S0>::x(r)) + PassSlot<S0>::a(r)] = v[p][r];
}
template <int NP, int S0>
__device__ __forceinline__ void smem_load(const u64 *smem, u64 (&v)[NP][8], int t) {
    const int base = swz(elem_index<S0>(t, 0));
#pragma unroll
    for (int p = 0; p < NP; p++)
#pragma unroll
        for (int r = 0; r < 8; r++) v[p][r] = smem[p * kN + (base ^ PassSlot<S0>::x(r)) + PassSlot<S0>::a(r)];
}

// ---------------------------------------------------------------- whole transforms on registers
// Forward NTT of NP polynomials.
//  in : v holds coefficients elem_index<0>(t, r) = r*512 + t   (natural order; small primes < 2^42, large < 2q)
//  out: v holds NTT values at positions elem_index<9>(t, r) = 8*t + r, reduced to [0, q) if kCanon
//       (else small primes < in + 60q, large primes < 8q).  Large-prime inputs must be < 2q.
template <class M, int NP, bool kCanon, bool kTrailSync = true>
__device__ __forceinline__ void ntt_forward(u64 (&v)[NP][8], u64 *smem, const ulonglong2 *__restrict__ tw, int t) {
    fwd_pass<M, NP, 0>(v, tw, pass_upper<0>(t));
    smem_store<NP, 0>(smem, v, t);
    __syncthreads();
    smem_load<NP, 3>(smem, v, t);
    fwd_pass<M, NP, 3>(v, tw, pass_upper<3>(t));
    smem_store<NP, 3>(smem, v, t);
    sync_group64(t);
    smem_load<NP, 6>(smem, v, t);
    fwd_pass<M, NP, 6>(v, tw, pass_upper<6>(t));
    smem_store<NP, 6>(smem, v, t);
    __syncwarp();
    smem_load<NP, 9>(smem, v, t);
    fwd_pass<M, NP, 9>(v, tw, pass_upper<9>(t));
    if constexpr (kCanon && !M::kDual) {
#pragma unroll
        for (int p = 0; p < NP; p++)
#pragma unroll
            for (int r = 0; r < 8; r++) v[p][r] = canon_k32<M>(v[p][r]);  // small: < 2^44; large: < 8q
    }
    if (kTrailSync) __syncthreads();  // smem may be reused by the caller
}

// Inverse NTT of NP polynomials.
//  in : v holds NTT values at positions 8*t + r, each < 2q (small primes: < 4q)
//  out: v holds coefficients r*512 + t, multiplied by the scalar sc (scw = sc * last-stage twiddle), in [0, q)
//       ([0, 2q) if !kCanon)
template <class M, int NP, bool kCanon = true, bool kTrailSync = true>
__device__ __forceinline__ void ntt_inverse(u64 (&v)[NP][8], u64 *smem, const ulonglong2 *__restrict__ tw, int t, const Shoup &sc,
                                            const Shoup &scw) {
    inv_pass<M, NP, 9, 0>(v, tw, pass_upper<9>(t));
    smem_store<NP, 9>(smem, v, t);
    __syncwarp();
    smem_load<NP, 6>(smem, v, t);
    inv_pass<M, NP, 6, 3>(v, tw, pass_upper<6>(t));
    smem_store<NP, 6>(smem, v, t);
    sync_group64(t);
    smem_load<NP, 3>(smem, v, t);
    inv_pass<M, NP, 3, 6>(v, tw, pass_upper<3>(t));
    smem_store<NP, 3>(smem, v, t);
    __syncthreads();
    smem_load<NP, 0>(smem, v, t);
    inv_pass<M, NP, 0, 9, true, kCanon>(v, tw, pass_upper<0>(t), &sc, &scw);
    if (kTrailSync) __syncthreads();
}

// ---------------------------------------------------------------- global <-> register helpers
// natural-order limb (4096 u64) -> registers in pass-0 layout (coalesced 8-byte accesses)
__device__ __forceinline__ void load_natural(const u64 *__restrict__ g, u64 (&v)[8], int t) {
#pragma unroll
    for (int r = 0; r < 8; r++) v[r] = g[r * kThreads + t];
}
__device__ __forceinline__ void store_natural(u64 *__restrict__ g, const u64 (&v)[8], int t) {
#pragma unroll
    for (int r = 0; r < 8; r++) g[r * kThreads + t] = v[r];
}
// bit-reversed-domain limb <-> registers in pass-9 layout (thread owns 8 consecutive values, 16-byte accesses)
__device__ __forceinline__ void load_chunk8(const u64 *__restrict__ g, u64 (&v)[8], int t) {
    const ulonglong2 *p = reinterpret_cast<const ulonglong2 *>(g + 8 * t);
#pragma unroll
    for (int r = 0; r < 4; r++) {
        ulonglong2 x = p[r];
        v[2 * r] = x.x;
        v[2 * r + 1] = x.y;
    }
}
__device__ __forceinline__ void load_chunk8_ldg(const u64 *__restrict__ g, u64 (&v)[8], int t) {
    const ulonglong2 *p = reinterpret_cast<const ulonglong2 *>(g + 8 * t);
#pragma unroll
    for (int r = 0; r < 4; r++) {
        ulonglong2 x = __ldg(p + r);
        v[2 * r] = x.x;
        v[2 * r + 1] = x.y;
    }
}
// The library's own NTT-domain scratch limbs (extended operands, key-switch digits: never seen outside) use a LANE-MAJOR chunk
// layout instead: pair j of thread t -- NTT positions 8t + 2j and 8t + 2j + 1 -- lives in 16-byte slot j * 512 + t, so a warp
// reads or writes one contiguous 512-byte run per instruction instead of 32 pieces of 16 bytes spread over 2 KiB (the
// transforms are L1-wavefront bound once the arithmetic is cheap).
constexpr int kLm = kThreads;  // slot distance between a thread's consecutive pairs
__device__ __forceinline__ const ulonglong2 *lm_ptr(const u64 *__restrict__ g, int t) { return reinterpret_cast<const ulonglong2 *>(g) + t; }
__device__ __forceinline__ void store_chunk8_lm(u64 *__restrict__ g, const u64 (&v)[8], int t) {
    ulonglong2 *p = reinterpret_cast<ulonglong2 *>(g) + t;
#pragma unroll
    for (int j = 0; j < 4; j++) p[j * kLm] = make_ulonglong2(v[2 * j], v[2 * j + 1]);
}
__device__ __forceinline__ void load_chunk8_lm(const u64 *__restrict__ g, u64 (&v)[8], int t) {
    const ulonglong2 *p = lm_ptr(g, t);
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const ulonglong2 x = p[j * kLm];
        v[2 * j] = x.x;
        v[2 * j + 1] = x.y;
    }
}
__device__ __forceinline__ void store_chunk8(u64 *__restrict__ g, const u64 (&v)[8], int t) {
    ulonglong2 *p = reinterpret_cast<ulonglong2 *>(g + 8 * t);
#pragma unroll
    for (int r = 0; r < 4; r++) p[r] = make_ulonglong2(v[2 * r], v[2 * r + 1]);
}

}  // namespace fheb
