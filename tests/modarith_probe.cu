// Contract probe for csrc/modarith.cuh and the butterflies of csrc/ntt.cuh (tests/test_modarith_contracts.py).
//
// Every primitive there states an input domain and a lazy, non-canonical output range, and the transforms chain those
// ranges without reducing in between: a result one q above its stated range is still congruent and breaks nothing until
// a later stage overflows a word.  This probe runs the COMPILED sm_100a primitives on crafted and top-of-domain operands
// and checks, per operand tuple, congruence against an independent exact reference (unsigned __int128 and %, never the
// primitive's own partial products) and the stated range.
//
//   modarith_probe --cpu            host checks: twiddle tables, DevConsts Shoup pairs, derived constants, bound table
//   modarith_probe [--case a,b,..]  GPU cases (all, or those whose name starts with one of the prefixes)
//
// Each case prints "case <name> evaluated=<n> cong_fail=<n> range_fail=<n> max_out/q=<x>"; on a failure it prints up to
// eight failing tuples ("in" = operands, then the output and the limit it broke) and the probe exits nonzero.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "context.h"
namespace fheb {
namespace {  // internal linkage: the probe's own copies, distinct from kernels.o's
__constant__ DevTwLow ktl;  // read by ntt.cuh's ldtw, which the probe does not call
__constant__ DevConsts kc;
}  // namespace
}  // namespace fheb
#include "ntt.cuh"

using namespace fheb;
typedef unsigned __int128 u128;

// ---------------------------------------------------------------- the bound table (ntt.cuh, fwd_bfly / inv_bfly / ntt_*)
// Per stage G: the bound of the values a stage takes and of the two values it leaves, in units of the modulus.
//  small primes, forward : inputs < 2^42 (ntt_forward) + 5q per stage (T = wY in [0, 5q))
//  61-bit primes, forward: 2q -> 4q -> 6q -> 8q, X folded below 2q on stages 3, 6, 9 (Y is taken at any 64-bit value)
//  small primes, inverse : inputs < 4q 2^G, X out < 4q 2^(G+1), Y out < 4q
//  61-bit primes, inverse: even stages 2q -> (X 4q, Y 2q), odd stages 4q -> (X 2q, Y 2q)
//  dual limbs: forward [0, 4s) -> [0, 4s), inverse [0, 2s) -> [0, 2s); last inverse stage [0, 2s) -> [0, 2s) or canonical
constexpr u64 kFwdSmallBase = 1ull << 42;
__host__ __device__ constexpr u64 fwd_in(u64 q, bool small, int G) {
    constexpr int kSmall[12] = {0, 5, 10, 15, 20, 25, 30, 35, 40, 45, 50, 55};  // + kFwdSmallBase
    constexpr int kLarge[12] = {2, 4, 6, 8, 4, 6, 8, 4, 6, 8, 4, 6};
    return small ? kFwdSmallBase + kSmall[G] * q : kLarge[G] * q;
}
__host__ __device__ constexpr u64 fwd_out(u64 q, bool small, int G) {
    constexpr int kSmall[12] = {5, 10, 15, 20, 25, 30, 35, 40, 45, 50, 55, 60};  // + kFwdSmallBase
    constexpr int kLarge[12] = {4, 6, 8, 4, 6, 8, 4, 6, 8, 4, 6, 8};
    return small ? kFwdSmallBase + kSmall[G] * q : kLarge[G] * q;
}
__host__ __device__ constexpr u64 inv_in(u64 q, bool small, int G) { return small ? (4 * q) << G : (G % 2 ? 4 : 2) * q; }
__host__ __device__ constexpr u64 inv_out_x(u64 q, bool small, int G) { return small ? (4 * q) << (G + 1) : (G % 2 ? 2 : 4) * q; }
__host__ __device__ constexpr u64 inv_out_y(u64 q, bool small, int) { return small ? 4 * q : 2 * q; }

// ---------------------------------------------------------------- results
constexpr int kSlots = 8;
struct Stats {
    unsigned long long evaluated, cong, range, maxfx;  // maxfx: largest out / unit, in 1/1024
    unsigned nrec;
    u64 rec[kSlots][6];  // up to four operands, output, limit
};

__device__ void verdict(Stats *st, u64 &mx, bool cong_ok, u64 out, u64 lim, u64 unit, u64 a, u64 b = 0, u64 c = 0, u64 d = 0) {
    const bool range_ok = lim == 0 || out < lim;  // lim 0: no range stated
    if (unit) {
        const u128 r = ((u128)out << 10) / unit;
        const u64 f = r >> 64 ? ~0ull : (u64)r;
        if (f > mx) mx = f;
    }
    if (cong_ok && range_ok) return;
    if (!cong_ok) atomicAdd(&st->cong, 1ull);
    if (!range_ok) atomicAdd(&st->range, 1ull);
    const unsigned slot = min(atomicAdd(&st->nrec, 1u), (unsigned)kSlots);
    if (slot < kSlots) {
        u64 *r = st->rec[slot];
        r[0] = a, r[1] = b, r[2] = c, r[3] = d, r[4] = out, r[5] = lim;
    }
}

template <class C>
__global__ void __launch_bounds__(256) k_case(C c, u64 n, Stats *st) {
    u64 cnt = 0, mx = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        c(i, st, mx);
        cnt++;
    }
    atomicAdd(&st->evaluated, (unsigned long long)cnt);
    atomicMax(&st->maxfx, (unsigned long long)mx);
}

// ---------------------------------------------------------------- operands
__host__ __device__ inline u64 mix(u64 x) {  // splitmix64
    x += 0x9e3779b97f4a7c15ull;
    x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
    x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}
__device__ inline int nbits(u64 top) { return 64 - __clzll(top | 1); }  // top < 2^nbits
__device__ inline u64 uniform(u64 r, u64 top) { return top == ~0ull ? r : __umul64hi(r, top + 1); }

// edge j (0..15) of [0, top]: the top and just below it, multiples of q and their neighbours, powers of two, all-ones low words
__device__ u64 edge(int j, u64 top, u64 q) {
    const int nb = nbits(top);
    u64 v;
    switch (j & 15) {
        case 0: v = top; break;
        case 1: v = top - 1; break;
        case 2: v = q - 1; break;
        case 3: v = q; break;
        case 4: v = 2 * q - 1; break;
        case 5: v = top / q * q; break;
        case 6: v = top / q * q - 1; break;
        case 7: v = 1ull << (nb - 1); break;
        case 8: v = (1ull << (nb - 1)) - 1; break;
        case 9: v = top >> 32 ? ((top >> 32) << 32) - 1 : top; break;
        case 10: v = 0; break;
        case 11: v = 1; break;
        case 12: v = top - q + 1; break;
        case 13: v = top - (1ull << (nb / 2)); break;
        case 14: v = 4 * q - 1; break;
        default: v = top >> 1; break;
    }
    return v > top ? top : v;  // also catches the wrapped ones
}
// random operand in [0, top], shaped toward the top of the domain
__device__ u64 pick(u64 r, u64 top, u64 q) {
    const u64 r2 = mix(r);
    const int nb = nbits(top);
    u64 v;
    switch (r & 7) {
        case 0: case 1: v = uniform(r2, top); break;
        case 2: v = top - (r2 & 255); break;
        case 3: v = top - ((1ull << (r2 % nb)) - 1); break;
        case 4: v = uniform(r2, top) | 0xffffffffull; break;
        case 5: v = (1 + uniform(r2 >> 8, top / q)) * q - (r2 & 1); break;
        case 6: v = (1ull << (r2 % nb)) - ((r2 >> 8) & 1); break;
        default: v = r2 & 0xffff; break;
    }
    return v > top ? uniform(r2, top) : v;
}
// operand k of evaluation i, `round` = how often the case's constant list has been cycled: the first 16 rounds take every
// operand from the same edge (so the all-maximal tuple is among them), the next 16 mix edges, the rest are random
__device__ u64 operand(u64 seed, u64 i, int k, u64 round, u64 top, u64 q) {
    if (round < 16) return edge((int)round, top, q);
    if (round < 32) return edge((int)round + 5 * k, top, q);
    return pick(mix(seed ^ mix(i * 8 + k)), top, q);
}
__device__ inline u64 mm(u64 a, u64 b, u64 q) { return (u64)((u128)a * b % q); }

// ---------------------------------------------------------------- cases: Shoup products
// K = 0, 1, 2: shoup_acc<M, K>; 3: shoup_lazy; 4: shoup.  w: every twiddle of M plus the DevConsts pairs of M.
template <class M, int K>
struct ShoupCase {
    const ulonglong2 *w;
    u64 nw, seed;
    __device__ void operator()(u64 i, Stats *st, u64 &mx) const {
        const ulonglong2 p = w[i % nw];
        const u64 round = i / nw;
        const u64 x = operand(seed, i, 0, round, K == 2 ? (1ull << 44) - 1 : ~0ull, M::q);
        const u64 acc = K <= 2 ? operand(seed, i, 1, round, M::kSmall ? (1ull << 44) - 1 : (1ull << 62) - 1, M::q) : 0;
        u64 r, lim;
        if constexpr (K <= 2) {
            r = shoup_acc<M, K>(acc, x, p.x, p.y) - acc;  // the value added to acc
            lim = (K == 0 ? 2 : K == 1 ? 4 : 5) * M::q;
        } else if constexpr (K == 3) {
            r = shoup_lazy<M>(x, p.x, p.y), lim = M::two_q;
        } else {
            r = shoup<M>(x, p.x, p.y), lim = M::q;
        }
        verdict(st, mx, r % M::q == mm(x, p.x, M::q), r, lim, M::q, x, p.x, p.y, acc);
    }
};

// ---------------------------------------------------------------- cases: dual-limb (32-bit) primitives
struct Shoup32Case {  // every 32-bit x
    u32 w, ws, s;
    __device__ void operator()(u64 i, Stats *st, u64 &mx) const {
        const u32 x = (u32)i, out = shoup32(x, w, ws, s);
        verdict(st, mx, out % s == (u64)x * w % s, out, 2ull * s, s, x, w, ws);
    }
};
struct Barrett61Case {
    u32 mu, s;
    u64 seed;
    __device__ void operator()(u64 i, Stats *st, u64 &mx) const {
        const u64 V = operand(seed, i, 0, i, (1ull << 61) - 1, s);
        const u32 out = barrett61(V, mu, s);
        verdict(st, mx, out % s == V % s, out, 4ull * s, s, V, mu);
    }
};
template <int NP>
struct DualMulsumCase {
    u32 mu, s;
    u64 seed;
    __device__ void operator()(u64 i, Stats *st, u64 &mx) const {
        u32 x[NP], y[NP];
        u64 ref = 0;
        for (int k = 0; k < NP; k++) {
            x[k] = (u32)operand(seed, i, 2 * k, i, 4ull * s - 1, s);
            y[k] = (u32)operand(seed, i, 2 * k + 1, i, 4ull * s - 1, s);
            ref += (u64)(x[k] % s) * (y[k] % s) % s;
        }
        const u32 out = dual_mulsum<NP>(x, y, s, mu);
        verdict(st, mx, out % s == ref % s, out, 2ull * s, s, x[0], y[0], NP == 2 ? x[1] : 0, NP == 2 ? y[1] : 0);
    }
};

// ---------------------------------------------------------------- cases: WideSum
// One weight set: T add32 weights, S add_small weights, and (kLo) a constant added to `lo` with one more operand < q, the
// shapes k_floor_sk_d (T = 6 or 4, S = 1) and ks_finish_coeff_ksd (T = 6, S = 1; T = 7, S = 2, lo += c + ksHd) use.
struct WSet {
    u64 w[7], ws[2], h;
};
template <class M, int T, int S, bool kLo>
struct WideSumCase {
    const WSet *sets;
    u64 nsets, seed;
    __device__ void operator()(u64 i, Stats *st, u64 &mx) const {
        const WSet &ws = sets[i % nsets];
        const u64 round = i / nsets;
        WideSum<M> sum;
        u128 ref = 0;
        u64 x0 = 0;
        for (int k = 0; k < T; k++) {
            const u32 x = (u32)operand(seed, i, k, round, (1ull << 31) - 1, M::q);
            sum.add32(x, ws.w[k]);
            ref += (u128)x * ws.w[k];
            if (k == 0) x0 = x;
        }
        for (int k = 0; k < S; k++) {
            const u32 x = (u32)operand(seed, i, 8 + k, round, 255, M::q);
            sum.add_small(x, ws.ws[k]);
            ref += (u128)x * ws.ws[k];
        }
        u64 c = 0;
        if (kLo) {
            c = operand(seed, i, 12, round, M::q - 1, M::q);
            sum.lo += c + ws.h;
            ref += c + ws.h;
        }
        const u64 out = sum.value();
        verdict(st, mx, out == (u64)(ref % M::q) || (out >= M::q && out % M::q == (u64)(ref % M::q)), out, M::q, M::q, x0, ws.w[0], c, i % nsets);
    }
};

// ---------------------------------------------------------------- cases: variable products and reductions
template <class M, int NP>
struct MulsumCase {  // mulsum_small (36/37-bit, operands < 2^44) / mulsum_large (61-bit, operands < 2^61): [0, 2q)
    u64 seed;
    __device__ void operator()(u64 i, Stats *st, u64 &mx) const {
        constexpr u64 top = M::kSmall ? (1ull << 44) - 1 : (1ull << 61) - 1;
        u64 x[NP], y[NP];
        u128 ref = 0;
        for (int k = 0; k < NP; k++) {
            x[k] = operand(seed, i, 2 * k, i, top, M::q);
            y[k] = operand(seed, i, 2 * k + 1, i, top, M::q);
            ref += (u128)x[k] * y[k];
        }
        u64 out;
        if constexpr (M::kSmall)
            out = mulsum_small<M, NP>(x, y);
        else
            out = mulsum_large<M, NP>(x, y);
        verdict(st, mx, out % M::q == (u64)(ref % M::q), out, M::two_q, M::q, x[0], y[0], NP == 2 ? x[1] : 0, NP == 2 ? y[1] : 0);
    }
};
template <class M>
struct MulmodCase {  // canonical a b mod q
    u64 seed;
    __device__ void operator()(u64 i, Stats *st, u64 &mx) const {
        constexpr u64 top = M::kSmall ? (1ull << 44) - 1 : (1ull << 61) - 1;
        const u64 a = operand(seed, i, 0, i, top, M::q), b = operand(seed, i, 1, i, top, M::q);
        const u64 out = mulmod<M>(a, b);
        verdict(st, mx, out == mm(a, b, M::q), out, M::q, M::q, a, b);
    }
};
// fold / fold_k32 / canon / canon_k32 / reduce64 / addmod / submod at their stated domains
enum { kFold, kFoldK32, kCanon, kCanonK32, kReduce64, kAddmod, kSubmod };
template <class M, int F>
struct ReduceCase {
    u64 seed;
    // fold_k32 / canon_k32 need floor(x / 2^b) c < 2^32; canon needs fold(x) < 2q (small primes: x < 2^54)
    static constexpr u64 top = F == kFoldK32 || F == kCanonK32 ? (M::kSmall ? (1ull << 50) - 1 : ~0ull)
                               : F == kCanon               ? (M::kSmall ? (1ull << 54) - 1 : ~0ull)
                               : F >= kAddmod              ? M::q - 1
                                                           : ~0ull;
    __device__ void operator()(u64 i, Stats *st, u64 &mx) const {
        const u64 x = operand(seed, i, 0, i, top, M::q), y = operand(seed, i, 1, i, top, M::q);
        u64 out, lim = M::q, ref = x % M::q;
        if constexpr (F == kFold) out = fold<M>(x), lim = (1ull << M::kBits) + (M::kC << (64 - M::kBits));
        if constexpr (F == kFoldK32) out = fold_k32<M>(x), lim = (1ull << M::kBits) + (1ull << 32);
        if constexpr (F == kCanon) out = canon<M>(x);
        if constexpr (F == kCanonK32) out = canon_k32<M>(x);
        if constexpr (F == kReduce64) out = reduce64<M>(x);
        if constexpr (F == kAddmod) out = addmod<M>(x, y), ref = (x + y) % M::q;
        if constexpr (F == kSubmod) out = submod<M>(x, y), ref = (x + M::q - y) % M::q;
        const bool exact = F == kFold || F == kFoldK32 ? out % M::q == ref : out == ref;
        verdict(st, mx, exact, out, lim, M::q, x, F >= kAddmod ? y : 0);
    }
};
struct Mac128Case {  // (hi:lo) += a b, exactly, for any 64-bit operands
    u64 seed;
    __device__ void operator()(u64 i, Stats *st, u64 &mx) const {
        const u64 a = operand(seed, i, 0, i, ~0ull, 3), b = operand(seed, i, 1, i, ~0ull, 3);
        u64 lo = operand(seed, i, 2, i, ~0ull, 3), hi = operand(seed, i, 3, i, ~0ull, 3);
        const u128 ref = (((u128)hi << 64) | lo) + (u128)a * b;
        const u64 lo0 = lo, hi0 = hi;
        mac128(lo, hi, a, b);
        verdict(st, mx, lo == (u64)ref && hi == (u64)(ref >> 64), hi, 0, 0, a, b, lo0, hi0);
    }
};

// ---------------------------------------------------------------- cases: butterflies
// Kind 0: fwd_bfly<M, G>, 1: inv_bfly<M, G>, 2/3: inv_bfly_last<M, kCanon = false/true> with (N^-1, N^-1 w) or (N^-1 t, N^-1 t w).
// Inputs at the stage's input bound, twiddles of stage G (table indices [2^G, 2^(G+1))); outputs checked against the table.
template <class M, int G, int kKind>
struct BflyCase {
    const ulonglong2 *tw;
    Shoup sc[2], scw[2];
    u64 seed;
    __device__ void operator()(u64 i, Stats *st, u64 &mx) const {
        constexpr u64 q = M::q;
        constexpr bool sm = M::kSmall;
        const int j = kKind == 0 || kKind == 1 ? (1 << G) + (int)(i & ((1u << G) - 1)) : 1;
        const u64 round = kKind <= 1 ? i >> G : i >> 1;
        const u64 in = kKind == 0 ? fwd_in(q, sm, G) : kKind == 1 ? inv_in(q, sm, G) : inv_in(q, sm, 11);
        const u64 X = operand(seed, i, 0, round, in - 1, q), Y = operand(seed, i, 1, round, in - 1, q);
        u64 x = X, y = Y, rx, ry, limx, limy, w = 0;
        if constexpr (kKind == 0) {
            w = tw[j].x;
            fwd_bfly<M, G>(x, y, tw[j].x, tw[j].y);
            rx = (X % q + mm(w, Y % q, q)) % q, ry = (X % q + q - mm(w, Y % q, q)) % q;
            limx = limy = fwd_out(q, sm, G);
        } else if constexpr (kKind == 1) {
            w = tw[j].x;
            inv_bfly<M, G>(x, y, tw[j].x, tw[j].y);
            rx = (X % q + Y % q) % q, ry = mm(w, (X % q + q - Y % q) % q, q);
            limx = inv_out_x(q, sm, G), limy = inv_out_y(q, sm, G);
        } else {
            const Shoup s = sc[i & 1], sw = scw[i & 1];
            w = s.w;
            inv_bfly_last<M, kKind == 3>(x, y, s, sw);
            rx = mm(s.w, (X % q + Y % q) % q, q), ry = mm(sw.w, (X % q + q - Y % q) % q, q);
            limx = limy = kKind == 3 ? q : 2 * q;
        }
        verdict(st, mx, x % q == rx, x, limx, q, X, Y, w, 0);
        verdict(st, mx, y % q == ry, y, limy, q, X, Y, w, 1);
    }
};
template <int D, int G, int kKind>
struct DualBflyCase {  // the same on both 32-bit lanes of ModDual<D>
    const ulonglong2 *tw;
    Shoup sc[2], scw[2];
    u64 seed;
    __device__ void operator()(u64 i, Stats *st, u64 &mx) const {
        using M = ModDual<D>;
        const int j = kKind <= 1 ? (1 << G) + (int)(i & ((1u << G) - 1)) : 1;
        const u64 round = kKind <= 1 ? i >> G : i >> 1;
        const u32 s[2] = {M::s0, M::s1};
        const u64 in = kKind == 0 ? 4 : 2;  // units of s
        u32 X[2], Y[2];
        for (int l = 0; l < 2; l++) {
            X[l] = (u32)operand(seed, i, 2 * l, round, in * s[l] - 1, s[l]);
            Y[l] = (u32)operand(seed, i, 2 * l + 1, round, in * s[l] - 1, s[l]);
        }
        u64 x = pack64(X[0], X[1]), y = pack64(Y[0], Y[1]), w = 0, wx = 0;
        if constexpr (kKind == 0) {
            w = tw[j].x, wx = w;
            fwd_bfly<M, G>(x, y, tw[j].x, tw[j].y);
        } else if constexpr (kKind == 1) {
            w = tw[j].x, wx = w;
            inv_bfly<M, G>(x, y, tw[j].x, tw[j].y);
        } else {
            const Shoup a = sc[i & 1], b = scw[i & 1];
            w = b.w, wx = a.w;
            inv_bfly_last<M, kKind == 3>(x, y, a, b);
        }
        for (int l = 0; l < 2; l++) {
            const u64 sl = s[l], wl = (w >> (32 * l)) & 0xffffffffu, wxl = (wx >> (32 * l)) & 0xffffffffu;
            const u32 ox = (u32)(x >> (32 * l)), oy = (u32)(y >> (32 * l));
            const u64 a = X[l] % sl, b = Y[l] % sl;
            u64 rx, ry, limx, limy;
            if (kKind == 0) rx = (a + wl * b) % sl, ry = (a + sl * sl - wl * b % sl) % sl, limx = limy = 4 * sl;
            else if (kKind == 1) rx = (a + b) % sl, ry = wl * ((a + sl - b) % sl) % sl, limx = limy = 2 * sl;
            else rx = wxl * ((a + b) % sl) % sl, ry = wl * ((a + sl - b) % sl) % sl, limx = limy = kKind == 3 ? sl : 2 * sl;
            verdict(st, mx, ox % sl == rx, ox, limx, sl, X[l], Y[l], wl, 2 * l);
            verdict(st, mx, oy % sl == ry, oy, limy, sl, X[l], Y[l], wl, 2 * l + 1);
        }
    }
};

// ---------------------------------------------------------------- host side
static int g_failed = 0;
static std::vector<std::string> g_only;
static std::vector<void *> g_mem;
static int g_cases = 0;

static void ck(cudaError_t e, const char *what) {
    if (e != cudaSuccess) {
        fprintf(stderr, "CUDA error in %s: %s\n", what, cudaGetErrorString(e));
        exit(2);
    }
}
template <class T>
static const T *upload(const std::vector<T> &v) {
    void *p = nullptr;
    ck(cudaMalloc(&p, v.size() * sizeof(T)), "cudaMalloc");
    ck(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice), "upload");
    g_mem.push_back(p);
    return (const T *)p;
}
static bool selected(const std::string &name) {
    if (g_only.empty()) return true;
    for (const auto &p : g_only)
        if (name.compare(0, p.size(), p) == 0) return true;
    return false;
}
template <class C>
static void run(const std::string &name, const C &c, u64 n) {
    if (!selected(name)) return;
    static Stats *st = nullptr;
    if (!st) ck(cudaMalloc(&st, sizeof(Stats)), "cudaMalloc(stats)");
    ck(cudaMemset(st, 0, sizeof(Stats)), "cudaMemset");
    k_case<<<148 * 8, 256>>>(c, n, st);
    ck(cudaGetLastError(), "launch");
    ck(cudaDeviceSynchronize(), name.c_str());
    Stats h;
    ck(cudaMemcpy(&h, st, sizeof(Stats), cudaMemcpyDeviceToHost), "download stats");
    const bool ok = h.evaluated == n && h.cong == 0 && h.range == 0;
    printf("case %s evaluated=%llu cong_fail=%llu range_fail=%llu max_out/q=%.4f%s\n", name.c_str(), h.evaluated, h.cong, h.range,
           h.maxfx / 1024.0, ok ? "" : "  FAILED");
    if (h.evaluated != n) printf("  evaluated %llu of %llu requested operands\n", h.evaluated, (unsigned long long)n);
    for (unsigned k = 0; k < h.nrec && k < (unsigned)kSlots; k++)
        printf("  in=[%#llx, %#llx, %#llx, %#llx] out=%#llx limit=%#llx\n", (unsigned long long)h.rec[k][0], (unsigned long long)h.rec[k][1],
               (unsigned long long)h.rec[k][2], (unsigned long long)h.rec[k][3], (unsigned long long)h.rec[k][4], (unsigned long long)h.rec[k][5]);
    g_failed += !ok;
    g_cases++;
}

static const char *const kModName[kNumMod] = {"q0", "q1", "P", "b0", "b1", "msk"};

// every 64-bit Shoup pair of DevConsts with the modulus its call sites use, and the 32-bit (lane) pairs with theirs
struct Pair64 {
    std::string name;
    u64 w, ws, m;
};
struct Pair32 {
    std::string name;
    u32 w, ws, s;
};
static std::vector<Pair64> pairs64(const DevConsts &c) {
    const u64 q[2] = {kModulus[MQ0], kModulus[MQ1]}, bsk[3] = {kModulus[MB0], kModulus[MB1], kModulus[MSK]};
    const u64 km[3] = {kModulus[MQ0], kModulus[MQ1], kModulus[MP]};
    std::vector<Pair64> v;
    auto add = [&](std::string n, const Shoup &s, u64 m) { v.push_back({n, s.w, s.ws, m}); };
    for (int mi = 0; mi < kNumMod; mi++) {
        const std::string i = "[" + std::to_string(mi) + "]";
        add("ninv" + i, c.ninv[mi], kModulus[mi]), add("ninv_t" + i, c.ninv_t[mi], kModulus[mi]);
        add("ninv_w" + i, c.ninv_w[mi], kModulus[mi]), add("ninv_t_w" + i, c.ninv_t_w[mi], kModulus[mi]);
    }
    for (int l = 0; l < 2; l++) {
        const std::string L = "[" + std::to_string(l) + "]";
        add("ext_in" + L, c.ext_in[l], q[l]), add("inv_punct_q" + L, c.inv_punct_q[l], q[l]);
        add("Bq" + L, c.Bq[l], q[l]), add("nBq" + L, c.nBq[l], q[l]), add("crtNB" + L, c.crtNB[l], q[l]);
        add("inv_P_mod_q" + L, c.inv_P_mod_q[l], q[l]), add("crt_inv" + L, c.crt_inv[l], q[l]);
        add("skV" + L, Shoup{c.skV[l], c.skVs[l]}, bsk[l]);
        for (int j = 0; j < 2; j++) add("pBq[" + std::to_string(j) + "]" + L, c.pBq[j][l], q[l]);
        for (int i = 0; i < 3; i++) add("crtK[" + std::to_string(i) + "]" + L, c.crtK[i][l], q[l]);
        for (int i = 0; i < 6; i++) add("d_K[" + std::to_string(i) + "]" + L, c.d_K[i][l], q[l]);
        for (int i = 0; i < 4; i++) add("d_P[" + std::to_string(i) + "]" + L, c.d_P[i][l], q[l]);
    }
    add("alK2", Shoup{c.alK2, c.alK2s}, bsk[2]), add("nib", c.nib, bsk[2]);
    for (int i = 0; i < 3; i++) add("crt3[" + std::to_string(i) + "]", c.crt3[i], bsk[i]);
    for (int m = 0; m < 3; m++) {
        add("lk_C[" + std::to_string(m) + "]", c.lk_C[m], km[m]);
        for (int i = 0; i < 6; i++) add("ksK[" + std::to_string(i) + "][" + std::to_string(m) + "]", c.ksK[i][m], km[m]);
    }
    return v;
}
static std::vector<Pair32> pairs32(const DevConsts &c) {
    std::vector<Pair32> v;
    for (int i = 0; i < 6; i++) v.push_back({"d_C[" + std::to_string(i) + "]", c.d_C[i], c.d_Cs[i], kDualPrime[i]});
    for (int i = 0; i < 4; i++) v.push_back({"d_W[" + std::to_string(i) + "]", c.d_W[i], c.d_Ws[i], kDualPrime[i]});
    for (int m = 0; m < 3; m++)
        for (int i = 0; i < 6; i++)
            v.push_back({"lk_R[" + std::to_string(m) + "][" + std::to_string(i) + "]", c.lk_R[m][i], c.lk_Rs[m][i], kDualPrime[i]});
    const Shoup *packed[4] = {c.d_ninv_t, c.d_ninv_t_w, c.d_ninv, c.d_ninv_w};
    const char *pn[4] = {"d_ninv_t", "d_ninv_t_w", "d_ninv", "d_ninv_w"};
    for (int k = 0; k < 4; k++)
        for (int d = 0; d < kNumDual; d++)
            for (int l = 0; l < 2; l++)
                v.push_back({std::string(pn[k]) + "[" + std::to_string(d) + "].lane" + std::to_string(l), (u32)(packed[k][d].w >> (32 * l)),
                             (u32)(packed[k][d].ws >> (32 * l)), kDualPrime[2 * d + l]});
    return v;
}

// ---------------------------------------------------------------- host checks (--cpu)
static long g_host_fail = 0;
#define HCHECK(cond, ...)                                          \
    do {                                                           \
        if (!(cond) && g_host_fail++ < 16) {                       \
            printf("host check failed (%s): ", #cond);             \
            printf(__VA_ARGS__);                                   \
            printf("\n");                                          \
        }                                                          \
    } while (0)

static u64 hmm(u64 a, u64 b, u64 q) { return (u64)((u128)a * b % q); }
static u64 hpow(u64 b, u64 e, u64 q) {
    u64 r = 1;
    for (; e; e >>= 1, b = hmm(b, b, q))
        if (e & 1) r = hmm(r, b, q);
    return r;
}
static int bitrev12(int x) {
    int r = 0;
    for (int i = 0; i < kLogN; i++) r = (r << 1) | ((x >> i) & 1);
    return r;
}
static u64 q64(u64 w, u64 m) { return (u64)(((u128)w << 64) / m); }
static u32 q32(u32 w, u32 s) { return (u32)(((u64)w << 32) / s); }

static void host_checks(const HostContext &H) {
    // twiddle tables: (w, ws) pairs, the pass-9 slot-major copy as ldtw reads it, rp[bitrev(i)] = psi^i with psi^N = -1
    long pairs = 0;
    for (int ti = 0; ti < kNumTab; ti++) {
        const bool dual = ti >= kNumMod;
        for (int inv = 0; inv < 2; inv++) {
            const std::vector<ulonglong2> &tab = inv ? H.twi[ti] : H.twf[ti];
            HCHECK(tab.size() == (size_t)kTwEntries, "table %d/%d has %zu entries", ti, inv, tab.size());
            if (tab.size() != (size_t)kTwEntries) continue;
            for (int k = 0; k < kTwEntries; k++) {
                if (!dual) {
                    const u64 q = kModulus[ti];
                    HCHECK(tab[k].x < q && tab[k].y == q64(tab[k].x, q), "tw%c[%d][%d] = (%#llx, %#llx)", inv ? 'i' : 'f', ti, k,
                           (unsigned long long)tab[k].x, (unsigned long long)tab[k].y);
                    pairs++;
                } else
                    for (int l = 0; l < 2; l++) {
                        const u32 s = kDualPrime[2 * (ti - kNumMod) + l], w = (u32)(tab[k].x >> (32 * l)), ws = (u32)(tab[k].y >> (32 * l));
                        HCHECK(w < s && ws == q32(w, s), "tw%c[%d][%d] lane %d = (%#x, %#x)", inv ? 'i' : 'f', ti, k, l, w, ws);
                        pairs++;
                    }
            }
            std::vector<int> hit(kTwPass9, 0);
            for (int i = 512; i < kN; i++) {  // ntt.cuh ldtw, S0 == 9
                const int lvl = i >= 2048 ? 2 : (i >= 1024 ? 1 : 0);
                const int t = (i - (512 << lvl)) >> lvl, h = i & ((1 << lvl) - 1);
                const int slot = ((1 << lvl) - 1 + h) * 512 + t;
                HCHECK(slot >= 0 && slot < kTwPass9, "pass-9 slot %d of entry %d", slot, i);
                if (slot < 0 || slot >= kTwPass9) continue;
                hit[slot]++;
                HCHECK(tab[kN + slot].x == tab[i].x && tab[kN + slot].y == tab[i].y, "table %d/%d pass-9 slot %d != entry %d", ti, inv, slot, i);
            }
            for (int s = 0; s < kTwPass9; s++) HCHECK(hit[s] == 1, "table %d/%d pass-9 slot %d read %d times", ti, inv, s, hit[s]);
        }
        for (int l = 0; l < (dual ? 2 : 1); l++) {
            const int sh = dual ? 32 * l : 0;
            const u64 q = dual ? kDualPrime[2 * (ti - kNumMod) + l] : kModulus[ti], mask = dual ? 0xffffffffull : ~0ull;
            auto f = [&](int k) { return (H.twf[ti][k].x >> sh) & mask; };
            auto g = [&](int k) { return (H.twi[ti][k].x >> sh) & mask; };
            const u64 psi = f(bitrev12(1));
            HCHECK(hpow(psi, kN, q) == q - 1, "table %d lane %d: psi^N != -1", ti, l);
            u64 pw = 1;
            for (int i = 0; i < kN; i++, pw = hmm(pw, psi, q)) {
                HCHECK(f(bitrev12(i)) == pw, "table %d lane %d: rp[bitrev(%d)] != psi^%d", ti, l, i, i);
                HCHECK(hmm(f(bitrev12(i)), g(bitrev12(i)), q) == 1, "table %d lane %d: twi[%d] is not the inverse", ti, l, bitrev12(i));
            }
        }
    }
    printf("host twiddle_pairs=%ld\n", pairs);

    // DevConsts Shoup pairs against the modulus of their call sites; the N^-1 scalings
    const DevConsts &c = H.dc;
    const auto p64 = pairs64(c);
    const auto p32 = pairs32(c);
    for (const auto &p : p64) HCHECK(p.w < p.m && p.ws == q64(p.w, p.m), "%s = (%#llx, %#llx)", p.name.c_str(), (unsigned long long)p.w, (unsigned long long)p.ws);
    for (const auto &p : p32) HCHECK(p.w < p.s && p.ws == q32(p.w, p.s), "%s = (%#x, %#x)", p.name.c_str(), p.w, p.ws);
    for (int mi = 0; mi < kNumMod; mi++) {
        const u64 m = kModulus[mi], wl = H.twi[mi][1].x;
        HCHECK(hmm(c.ninv[mi].w, kN, m) == 1, "ninv[%d]", mi);
        HCHECK(c.ninv_t[mi].w == hmm(c.ninv[mi].w, kT % m, m), "ninv_t[%d]", mi);
        HCHECK(c.ninv_w[mi].w == hmm(c.ninv[mi].w, wl, m) && c.ninv_t_w[mi].w == hmm(c.ninv_t[mi].w, wl, m), "ninv*_w[%d]", mi);
    }
    for (int d = 0; d < kNumDual; d++)
        for (int l = 0; l < 2; l++) {
            const u64 s = kDualPrime[2 * d + l], wl = (H.twi[kNumMod + d][1].x >> (32 * l)) & 0xffffffffu;
            auto lane = [&](const Shoup &x) { return (x.w >> (32 * l)) & 0xffffffffu; };
            HCHECK(hmm(lane(c.d_ninv[d]), kN, s) == 1 && lane(c.d_ninv_t[d]) == hmm(lane(c.d_ninv[d]), kT, s), "d_ninv[%d] lane %d", d, l);
            HCHECK(lane(c.d_ninv_w[d]) == hmm(lane(c.d_ninv[d]), wl, s) && lane(c.d_ninv_t_w[d]) == hmm(lane(c.d_ninv_t[d]), wl, s),
                   "d_ninv*_w[%d] lane %d", d, l);
        }
    printf("host devconsts_pairs64=%zu devconsts_pairs32=%zu\n", p64.size(), p32.size());

    // derived reduction constants
    for (int i = 0; i < 2 * kNumDual; i++) {
        const u64 s = kDualPrime[i];
        HCHECK(c.d_mu61[i] == (1ull << 61) / s && c.d_R48[i] == (1ull << 48) / s, "d_mu61 / d_R48 [%d]", i);
        HCHECK(c.d_R32[i] == (1ull << 32) % s && c.d_R61[i] == (1ull << 61) % s, "d_R32 / d_R61 [%d]", i);
        if (i < 4) HCHECK(c.d_R58[i] == (1ull << 58) % s, "d_R58[%d]", i);
    }
    const u128 all = ~(u128)0;  // floor(2^128 / q) = floor((2^128 - 1) / q): q is odd
    auto ratio = [&](u64 q, u64 r1, u64 r0, u64 C, int bits, bool small) {
        HCHECK(r1 == (u64)(all / q >> 64) && r0 == (u64)(all / q), "barrett_ratio(%#llx)", (unsigned long long)q);
        HCHECK(q == (1ull << bits) - C && C < (1u << 19) && q >> (bits - 1) == 1 && small == (q < (1ull << 40)), "Mod<%#llx> shape",
               (unsigned long long)q);
    };
    ratio(Mod<0>::q, Mod<0>::r1, Mod<0>::r0, Mod<0>::kC, Mod<0>::kBits, Mod<0>::kSmall);
    ratio(Mod<1>::q, Mod<1>::r1, Mod<1>::r0, Mod<1>::kC, Mod<1>::kBits, Mod<1>::kSmall);
    ratio(Mod<2>::q, Mod<2>::r1, Mod<2>::r0, Mod<2>::kC, Mod<2>::kBits, Mod<2>::kSmall);
    ratio(Mod<3>::q, Mod<3>::r1, Mod<3>::r0, Mod<3>::kC, Mod<3>::kBits, Mod<3>::kSmall);
    ratio(Mod<4>::q, Mod<4>::r1, Mod<4>::r0, Mod<4>::kC, Mod<4>::kBits, Mod<4>::kSmall);
    ratio(Mod<5>::q, Mod<5>::r1, Mod<5>::r0, Mod<5>::kC, Mod<5>::kBits, Mod<5>::kSmall);

    // the bound table composes inside the words and meets every primitive's precondition
    for (int mi = 0; mi < kNumMod; mi++) {
        const u64 q = kModulus[mi];
        const bool sm = q < (1ull << 40);
        for (int G = 0; G < 12; G++) {
            if (G < 11) HCHECK(fwd_out(q, sm, G) <= fwd_in(q, sm, G + 1), "forward stage %d -> %d, modulus %d", G, G + 1, mi);
            if (G < 11) HCHECK(inv_out_x(q, sm, G) <= inv_in(q, sm, G + 1) && inv_out_y(q, sm, G) <= inv_in(q, sm, G + 1), "inverse stage %d, modulus %d", G, mi);
            if (sm) HCHECK(fwd_in(q, sm, G) <= (1ull << 44), "forward stage %d: Y reaches 2^44 (shoup_acc<M, 2>), modulus %d", G, mi);
            if (sm) HCHECK((u128)2 * inv_in(q, sm, G) <= ((u128)1 << 51), "inverse stage %d: D reaches 2^51, modulus %d", G, mi);
            HCHECK(sm || (u128)8 * q < ((u128)1 << 64), "forward stage %d overflows a word, modulus %d", G, mi);
        }
        if (!sm) HCHECK(fwd_in(q, sm, 3) == 8 * q && (u128)8 * q < ((u128)1 << 64) && (1ull << 61) - 1 + 7 * Mod<3>::kC < 2 * q, "61-bit fold, modulus %d", mi);
        // ntt_forward's canonicalisation: fold_k32 of the last stage's outputs must be exact and < 2q
        const u64 top = fwd_out(q, sm, 11), C = (1ull << mod_bits(q)) - q;
        HCHECK((top >> mod_bits(q)) * C < (1ull << 32) && (1ull << mod_bits(q)) + (top >> mod_bits(q)) * C < 2 * q, "canon_k32 after forward, modulus %d", mi);
        if (sm) HCHECK(top < (1ull << 44), "small forward output %#llx >= 2^44, modulus %d", (unsigned long long)top, mi);
        // canon's domain (modarith.cuh): fold(x) < 2q for every small-prime x < 2^54
        if (sm) HCHECK((1ull << mod_bits(q)) - 1 + (((1ull << 54) - 1) >> mod_bits(q)) * C < 2 * q, "canon domain, modulus %d", mi);
    }
    for (int i = 0; i < 2 * kNumDual; i++) HCHECK((u64)4 * kDualPrime[i] < (1ull << 32), "4 s_%d does not fit a lane", i);
}

// ---------------------------------------------------------------- GPU cases
template <int MI>
static void shoup_cases(const HostContext &H, const std::vector<Pair64> &p64) {
    using M = Mod<MI>;
    std::vector<ulonglong2> w(H.twf[MI].begin(), H.twf[MI].begin() + kN);
    w.insert(w.end(), H.twi[MI].begin(), H.twi[MI].begin() + kN);
    for (const auto &p : p64)
        if (p.m == M::q) w.push_back(make_ulonglong2(p.w, p.ws));
    const ulonglong2 *dw = upload(w);
    const u64 nw = w.size(), n = nw * 512, seed = 0x5100 + MI;
    const std::string m = kModName[MI];
    run("shoup_acc0." + m, ShoupCase<M, 0>{dw, nw, seed}, n);
    if constexpr (M::kSmall) {
        run("shoup_acc1." + m, ShoupCase<M, 1>{dw, nw, seed + 16}, n);
        run("shoup_acc2." + m, ShoupCase<M, 2>{dw, nw, seed + 32}, n);
    }
    run("shoup_lazy." + m, ShoupCase<M, 3>{dw, nw, seed + 48}, n);
    run("shoup." + m, ShoupCase<M, 4>{dw, nw, seed + 64}, n);
}

template <class M>
static void widesum_cases(const HostContext &H, int mi) {
    const DevConsts &c = H.dc;
    const u64 q = M::q;
    const std::string m = kModName[mi];
    std::vector<WSet> s4, s6, s7;
    WSet top{};  // the all-maximal weights
    for (auto &w : top.w) w = q - 1;
    top.ws[0] = top.ws[1] = top.h = q - 1;
    s4.push_back(top), s6.push_back(top), s7.push_back(top);
    if (mi < 2) {  // k_floor_sk_d and ks_finish_coeff_ksd, q-limb l = mi
        WSet a{}, b{}, d{};
        for (int i = 0; i < 6; i++) a.w[i] = c.d_K[i][mi].w, d.w[i] = c.ksKd[i][mi];
        a.ws[0] = c.d_KN[mi];
        for (int i = 0; i < 4; i++) b.w[i] = c.d_P[i][mi].w;
        b.ws[0] = c.d_NS4[mi];
        d.w[6] = c.ksNd[mi], d.ws[0] = c.ksKNd[mi], d.ws[1] = c.ksNd30[mi], d.h = c.ksHd[mi];
        s6.push_back(a), s4.push_back(b), s7.push_back(d);
    } else {  // ks_finish_coeff_ksd, U mod P
        WSet a{};
        for (int i = 0; i < 6; i++) a.w[i] = c.ksK[i][2].w;
        a.ws[0] = c.ksKN[2];
        s6.push_back(a);
    }
    for (int r = 0; r < 64; r++) {  // random weights < q
        WSet x{};
        u64 z = 0x3000 + 97 * mi + r;
        for (auto &w : x.w) w = (z = mix(z)) % q;
        for (auto &w : x.ws) w = (z = mix(z)) % q;
        x.h = (z = mix(z)) % q;
        s4.push_back(x), s6.push_back(x), s7.push_back(x);
    }
    const u64 n = 1ull << 22;
    run("widesum4." + m, WideSumCase<M, 4, 1, false>{upload(s4), s4.size(), 0x4400u + mi}, n);
    run("widesum6." + m, WideSumCase<M, 6, 1, false>{upload(s6), s6.size(), 0x4600u + mi}, n);
    run("widesum7." + m, WideSumCase<M, 7, 2, true>{upload(s7), s7.size(), 0x4700u + mi}, n);
}

template <int MI>
static void reduce_cases() {
    using M = Mod<MI>;
    const std::string m = kModName[MI];
    const u64 n = 1ull << 22, seed = 0x7000 + 16 * MI;
    if constexpr (M::kSmall) {
        run("mulsum_small1." + m, MulsumCase<M, 1>{seed}, n);
        run("mulsum_small2." + m, MulsumCase<M, 2>{seed + 1}, n);
    } else {
        run("mulsum_large1." + m, MulsumCase<M, 1>{seed}, n);
        run("mulsum_large2." + m, MulsumCase<M, 2>{seed + 1}, n);
    }
    run("mulmod." + m, MulmodCase<M>{seed + 2}, n);
    run("fold." + m, ReduceCase<M, kFold>{seed + 3}, n);
    run("fold_k32." + m, ReduceCase<M, kFoldK32>{seed + 4}, n);
    run("canon." + m, ReduceCase<M, kCanon>{seed + 5}, n);
    run("canon_k32." + m, ReduceCase<M, kCanonK32>{seed + 6}, n);
    run("reduce64." + m, ReduceCase<M, kReduce64>{seed + 7}, n);
    run("addmod." + m, ReduceCase<M, kAddmod>{seed + 8}, n);
    run("submod." + m, ReduceCase<M, kSubmod>{seed + 9}, n);
}

template <int MI, int G>
static void bfly_mod(const ulonglong2 *f, const ulonglong2 *i, const Shoup (&sc)[2], const Shoup (&scw)[2]) {
    using M = Mod<MI>;
    const std::string m = kModName[MI], g = ".G" + std::to_string(G);
    const u64 n = 1ull << 20;
    run("fwd_bfly." + m + g, BflyCase<M, G, 0>{f, {sc[0], sc[1]}, {scw[0], scw[1]}, 0x8000u + 32 * MI + G}, n);
    run("inv_bfly." + m + g, BflyCase<M, G, 1>{i, {sc[0], sc[1]}, {scw[0], scw[1]}, 0x9000u + 32 * MI + G}, n);
    if constexpr (G < 11) bfly_mod<MI, G + 1>(f, i, sc, scw);
}
template <int MI>
static void bfly_cases(const HostContext &H) {
    const ulonglong2 *f = upload(H.twf[MI]), *i = upload(H.twi[MI]);
    const DevConsts &c = H.dc;
    const Shoup sc[2] = {c.ninv[MI], c.ninv_t[MI]}, scw[2] = {c.ninv_w[MI], c.ninv_t_w[MI]};
    bfly_mod<MI, 0>(f, i, sc, scw);
    const std::string m = kModName[MI];
    run("inv_bfly_last." + m + ".lazy", BflyCase<Mod<MI>, 11, 2>{i, {sc[0], sc[1]}, {scw[0], scw[1]}, 0xa000u + MI}, 1ull << 20);
    run("inv_bfly_last." + m + ".canon", BflyCase<Mod<MI>, 11, 3>{i, {sc[0], sc[1]}, {scw[0], scw[1]}, 0xa100u + MI}, 1ull << 20);
}
template <int D, int G>
static void bfly_dual(const ulonglong2 *f, const ulonglong2 *i, const Shoup (&sc)[2], const Shoup (&scw)[2]) {
    const std::string m = "d" + std::to_string(D), g = ".G" + std::to_string(G);
    const u64 n = 1ull << 20;
    run("fwd_bfly." + m + g, DualBflyCase<D, G, 0>{f, {sc[0], sc[1]}, {scw[0], scw[1]}, 0xb000u + 32 * D + G}, n);
    run("inv_bfly." + m + g, DualBflyCase<D, G, 1>{i, {sc[0], sc[1]}, {scw[0], scw[1]}, 0xc000u + 32 * D + G}, n);
    if constexpr (G < 11) bfly_dual<D, G + 1>(f, i, sc, scw);
}
template <int D>
static void dual_cases(const HostContext &H) {
    const int ti = kNumMod + D;
    const ulonglong2 *f = upload(H.twf[ti]), *i = upload(H.twi[ti]);
    const DevConsts &c = H.dc;
    const Shoup sc[2] = {c.d_ninv_t[D], c.d_ninv[D]}, scw[2] = {c.d_ninv_t_w[D], c.d_ninv_w[D]};
    bfly_dual<D, 0>(f, i, sc, scw);
    const std::string m = "d" + std::to_string(D);
    run("inv_bfly_last." + m + ".lazy", DualBflyCase<D, 11, 2>{i, {sc[0], sc[1]}, {scw[0], scw[1]}, 0xd000u + D}, 1ull << 20);
    run("inv_bfly_last." + m + ".canon", DualBflyCase<D, 11, 3>{i, {sc[0], sc[1]}, {scw[0], scw[1]}, 0xd100u + D}, 1ull << 20);
}

static void gpu_cases(const HostContext &H) {
    ck(cudaMemcpyToSymbol(kc, &H.dc, sizeof(DevConsts)), "upload DevConsts");
    const auto p64 = pairs64(H.dc);
    shoup_cases<MQ0>(H, p64), shoup_cases<MQ1>(H, p64), shoup_cases<MP>(H, p64);
    shoup_cases<MB0>(H, p64), shoup_cases<MB1>(H, p64), shoup_cases<MSK>(H, p64);

    // 32-bit Shoup products: every x for the DevConsts pairs that reach shoup32 and for a sample of dual twiddles
    for (const auto &p : pairs32(H.dc))
        if ((p.name.compare(0, 1, "d") == 0 && p.name.compare(0, 6, "d_ninv") != 0) || p.name.compare(0, 4, "lk_R") == 0)
            run("shoup32." + p.name, Shoup32Case{p.w, p.ws, p.s}, 1ull << 32);
    for (int d = 0; d < kNumDual; d++)
        for (int l = 0; l < 2; l++)
            for (int inv = 0; inv < 2; inv++)
                for (int k : {1, kN - 1}) {
                    const ulonglong2 e = (inv ? H.twi : H.twf)[kNumMod + d][k];
                    run("shoup32.tw" + std::string(inv ? "i" : "f") + ".s" + std::to_string(2 * d + l) + "." + std::to_string(k),
                        Shoup32Case{(u32)(e.x >> (32 * l)), (u32)(e.y >> (32 * l)), kDualPrime[2 * d + l]}, 1ull << 32);
                }
    for (int i = 0; i < 2 * kNumDual; i++) {
        const std::string s = ".s" + std::to_string(i);
        run("barrett61" + s, Barrett61Case{H.dc.d_mu61[i], kDualPrime[i], 0x6100u + i}, 1ull << 24);
        run("dual_mulsum1" + s, DualMulsumCase<1>{H.dc.d_mu61[i], kDualPrime[i], 0x6200u + i}, 1ull << 24);
        run("dual_mulsum2" + s, DualMulsumCase<2>{H.dc.d_mu61[i], kDualPrime[i], 0x6300u + i}, 1ull << 24);
    }

    widesum_cases<Mod<MQ0>>(H, MQ0), widesum_cases<Mod<MQ1>>(H, MQ1), widesum_cases<Mod<MP>>(H, MP);
    reduce_cases<MQ0>(), reduce_cases<MQ1>(), reduce_cases<MP>(), reduce_cases<MB0>(), reduce_cases<MB1>(), reduce_cases<MSK>();
    run("mac128", Mac128Case{0x7777}, 1ull << 22);

    bfly_cases<MQ0>(H), bfly_cases<MQ1>(H), bfly_cases<MP>(H), bfly_cases<MB0>(H), bfly_cases<MB1>(H), bfly_cases<MSK>(H);
    dual_cases<0>(H), dual_cases<1>(H), dual_cases<2>(H);
}

int main(int argc, char **argv) {
    bool cpu = false;
    for (int a = 1; a < argc; a++) {
        if (!strcmp(argv[a], "--cpu")) {
            cpu = true;
        } else if (!strcmp(argv[a], "--case") && a + 1 < argc) {
            std::string s = argv[++a];
            for (size_t p = 0; p <= s.size();) {
                const size_t e = s.find(',', p) == std::string::npos ? s.size() : s.find(',', p);
                if (e > p) g_only.push_back(s.substr(p, e - p));
                p = e + 1;
            }
        } else {
            fprintf(stderr, "usage: %s [--cpu | --case prefix[,prefix...]]\n", argv[0]);
            return 2;
        }
    }
    const HostContext &H = HostContext::get();
    if (H.dc.opaque_zero != 0) {
        printf("DevConsts::opaque_zero is %u, not 0\n", H.dc.opaque_zero);
        return 1;
    }
    if (cpu) {
        host_checks(H);
        printf(g_host_fail ? "host FAILED (%ld)\n" : "host ok\n", g_host_fail);
        return g_host_fail ? 1 : 0;
    }
    gpu_cases(H);
    for (void *p : g_mem) cudaFree(p);
    if (g_cases == 0) {
        printf("no case selected\n");
        return 1;
    }
    printf(g_failed ? "gpu FAILED (%d of %d cases)\n" : "gpu ok (%d of %d cases failed)\n", g_failed, g_cases);
    return g_failed ? 1 : 0;
}
