// sunscreen's value <-> plaintext encodings on the GPU (value_kernels.h), restating encode_scalar / decode_scalar (codec.cpp):
//   k_encode_values : one thread per 8 coefficients of a row (one 16-byte store), zero tail included
//   k_decode_int    : one warp per op over the 64 (u64, i64) or 256 (u256) coefficients the host reads; the sums are mod 2^64 /
//                     2^256, so the shuffle reduction's order does not matter
//   k_decode_frac   : one thread per op.  The host's value is a floating-point sum in index order, so each thread adds its
//                     row's terms in that order with the host's roundings (no FMA contraction: __dmul_rn / __dadd_rn).  Terms
//                     with power < -1074 (indices 64 .. 3021) are exactly zero and are not read: adding +-0 to the running
//                     sum never changes it, because in round-to-nearest that sum is never -0.
// No grid dimension depends on n: every kernel strides over the batch, so n > 65,535 needs no chunking.
#include "kernels.h"
#include "value_kernels.h"

namespace fheb {

namespace {
enum : int { kU256 = 0, kU64 = 1, kI64 = 2, kFrac64 = 3 };
constexpr u32 kCutoff = (u32)(kT + 1) / 2;
constexpr int kChunks = kN / 8;       // uint4 chunks per plaintext row
constexpr int kFracLow = 3016 / 8;    // first chunk of the negative powers that can be nonzero: index 3022 is 2^-1074
constexpr int kBlock = 256;
constexpr size_t kMaxBlocks = 1 << 16;

unsigned grid_for(size_t threads) {
    size_t g = (threads + kBlock - 1) / kBlock;
    return (unsigned)(g < kMaxBlocks ? g : kMaxBlocks);
}

// encode_scalar's return for the op: 7 for a frac64 NaN, +-inf or |v| >= 2^64 (their rows stay zero), otherwise 0
template <int K>
__device__ __forceinline__ int encode_status(const u64 *w) {
    if (K != kFrac64) return 0;
    const int e = (int)((w[0] >> 52) & 0x7ff);
    return (e == 0x7ff || (e - 1023) + 1 > 64) ? 7 : 0;
}

// coefficient i of encode_scalar(kind, v) for an op whose status is 0; w points at the op's value words
template <int K>
__device__ __forceinline__ u32 encode_coef(const u64 *w, int i) {
    if (K == kU64) return i < 64 ? (u32)((w[0] >> i) & 1) : 0u;
    if (K == kU256) return i < 256 ? (u32)((w[0] >> (i & 63)) & 1) : 0u;  // w: the word that holds coefficient i
    if (K == kI64) {
        if (i >= 64) return 0u;
        const long long v = (long long)w[0];
        const u64 mag = v < 0 ? (u64)0 - (u64)v : (u64)v;
        const u32 bit = (u32)((mag >> i) & 1);
        return v < 0 ? bit * (u32)(kT - bit) : bit;
    }
    // frac64: mantissa bit k (0..52) has power bp = power - 52 + k, stored at bp or, negative, at N + bp with the sign flipped
    const u64 bits = w[0];
    const int e = (int)((bits >> 52) & 0x7ff);
    if (e == 0) return 0u;  // +-0 and subnormals encode to the zero row
    const int power = e - 1023;
    const int bp = i < 64 ? i : i - kN;
    const int k = bp - power + 52;
    if (k < 0 || k > 52) return 0u;
    const u64 mant = (bits & 0xFFFFFFFFFFFFFull) | (1ull << 52);
    const u32 bit = (u32)((mant >> k) & 1);
    const u32 sg = (u32)(bits >> 63) ^ (bp < 0 ? 1u : 0u);
    return sg == 0 ? bit : bit * (u32)(kT - 1);
}

template <int K>
__global__ void __launch_bounds__(kBlock) k_encode_values(const u64 *__restrict__ values, uint16_t *__restrict__ plain,
                                                          int32_t *__restrict__ status, size_t n) {
    const size_t total = n * kChunks;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const size_t row = t / kChunks;
        const int i0 = (int)(t % kChunks) * 8;
        // a chunk's 8 coefficients come from one value word: u256 chunks read word i0 / 64 (chunks past 256 are zero)
        const u64 w[1] = {K == kU256 ? (i0 < 256 ? __ldg(values + row * 4 + (i0 >> 6)) : 0ull) : __ldg(values + row)};
        const int st = encode_status<K>(w);
        u32 c[8];
#pragma unroll
        for (int j = 0; j < 8; j++) c[j] = st ? 0u : encode_coef<K>(w, i0 + j);
        const uint4 out = make_uint4(c[0] | (c[1] << 16), c[2] | (c[3] << 16), c[4] | (c[5] << 16), c[6] | (c[7] << 16));
        reinterpret_cast<uint4 *>(plain + row * kN)[i0 / 8] = out;
        if (status && i0 == 0) status[row] = st;
    }
}

// (1 << i) * c, or -(1 << i) * (t - c) for c >= the cutoff, mod 2^64 exactly as the host's wrapping arithmetic
__device__ __forceinline__ u64 int_term(u32 c, int i) {
    return c < kCutoff ? (u64)c << i : (u64)0 - ((kT - (u64)c) << i);
}

__device__ __forceinline__ void add256(u64 a[4], const u64 b[4]) {
    u64 carry = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const u64 s = a[k] + b[k];
        const u64 c1 = s < a[k];
        const u64 s2 = s + carry;
        carry = c1 | (s2 < s);
        a[k] = s2;
    }
}

__device__ __forceinline__ void sub256(u64 a[4], const u64 b[4]) {
    u64 borrow = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const u64 d = a[k] - b[k];
        const u64 b1 = a[k] < b[k];
        const u64 d2 = d - borrow;
        borrow = b1 | (d < borrow);
        a[k] = d2;
    }
}

template <int K>
__global__ void __launch_bounds__(kBlock) k_decode_int(const uint16_t *__restrict__ plain, u64 *__restrict__ values, size_t n) {
    const int lane = threadIdx.x & 31;
    const size_t warps = (size_t)gridDim.x * (blockDim.x / 32);
    for (size_t row = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / 32; row < n; row += warps) {
        const uint16_t *p = plain + row * kN;
        if (K == kU256) {
            // lane owns coefficients 8 lane .. 8 lane + 7: word w = lane / 8, shifts s .. s + 7 within it
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p) + lane);
            const u32 h[4] = {v.x, v.y, v.z, v.w};
            const int w = lane >> 3;
            u64 acc[4] = {0, 0, 0, 0};
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const u32 c = (h[j >> 1] >> (16 * (j & 1))) & 0xffff;
                const int s = (lane & 7) * 8 + j;
                const bool neg = c >= kCutoff;
                const u64 mag = neg ? kT - (u64)c : (u64)c;  // wraps for c > t, as the host's
                const u64 lo = mag << s, hi = s ? mag >> (64 - s) : 0;  // mag << (64 w + s), truncated to 256 bits
                const u64 term[4] = {w == 0 ? lo : 0, w == 1 ? lo : (w == 0 ? hi : 0), w == 2 ? lo : (w == 1 ? hi : 0),
                                     w == 3 ? lo : (w == 2 ? hi : 0)};
                if (neg) sub256(acc, term);
                else add256(acc, term);
            }
#pragma unroll
            for (int off = 16; off; off >>= 1) {
                u64 o[4];
#pragma unroll
                for (int k = 0; k < 4; k++) o[k] = __shfl_xor_sync(0xffffffffu, acc[k], off);
                add256(acc, o);
            }
            if (lane == 0)
#pragma unroll
                for (int k = 0; k < 4; k++) values[row * 4 + k] = acc[k];
        } else {
            const u32 v = __ldg(reinterpret_cast<const u32 *>(p) + lane);  // coefficients 2 lane, 2 lane + 1
            u64 acc = int_term(v & 0xffff, 2 * lane) + int_term(v >> 16, 2 * lane + 1);
#pragma unroll
            for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
            if (lane == 0) values[row] = acc;
        }
    }
}

// 2^p exactly, from its bit pattern: normal for p >= -1022, subnormal down to -1074, 0 below (what exp2 returns there)
__device__ __forceinline__ double pow2_exact(int p) {
    if (p >= -1022) return __longlong_as_double((long long)(p + 1023) << 52);
    if (p >= -1074) return __longlong_as_double(1ll << (p + 1074));
    return 0.0;
}

// val +/-= sign * c * 2^power as decode_scalar writes it, for coefficient c at index i
__device__ __forceinline__ double frac_step(double val, u32 c, int i) {
    const int p = i < 64 ? i : i - kN;
    const bool neg = c >= kCutoff;
    const double x = neg ? __ull2double_rn(kT - (u64)c) : __uint2double_rn(c);  // the host's (double)(t - c), wrapped for c > t
    const double m = __dmul_rn(x, pow2_exact(p));  // the product's one rounding (subnormal results only)
    return __dadd_rn(val, (p >= 0) != neg ? m : -m);
}

__device__ __forceinline__ double frac_chunk(double val, uint4 v, int i0) {
    const u32 h[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 8; j++) val = frac_step(val, (h[j >> 1] >> (16 * (j & 1))) & 0xffff, i0 + j);
    return val;
}

__global__ void __launch_bounds__(kBlock) k_decode_frac(const uint16_t *__restrict__ plain, double *__restrict__ values, size_t n) {
    for (size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (size_t)gridDim.x * blockDim.x) {
        const uint4 *p = reinterpret_cast<const uint4 *>(plain + row * kN);
        double val = 0.0;
#pragma unroll
        for (int k = 0; k < 8; k++) val = frac_chunk(val, __ldg(p + k), 8 * k);
#pragma unroll 4
        for (int k = kFracLow; k < kChunks; k++) val = frac_chunk(val, __ldg(p + k), 8 * k);
        values[row] = val;
    }
}
}  // namespace

bool value_kind_valid(int kind) { return kind >= kU256 && kind <= kFrac64; }

cudaError_t launch_encode_values(int kind, const void *values, uint16_t *plain, int32_t *status, size_t n, cudaStream_t s) {
    if (!value_kind_valid(kind)) return cudaErrorInvalidValue;
    if (n == 0) return cudaSuccess;
    const unsigned g = grid_for(n * kChunks);
    const u64 *v = static_cast<const u64 *>(values);
    switch (kind) {
        case kU256: k_encode_values<kU256><<<g, kBlock, 0, s>>>(v, plain, status, n); break;
        case kU64: k_encode_values<kU64><<<g, kBlock, 0, s>>>(v, plain, status, n); break;
        case kI64: k_encode_values<kI64><<<g, kBlock, 0, s>>>(v, plain, status, n); break;
        default: k_encode_values<kFrac64><<<g, kBlock, 0, s>>>(v, plain, status, n); break;
    }
    count_launches(1);
    return cudaGetLastError();
}

cudaError_t launch_decode_values(int kind, const uint16_t *plain, void *values, size_t n, cudaStream_t s) {
    if (!value_kind_valid(kind)) return cudaErrorInvalidValue;
    if (n == 0) return cudaSuccess;
    switch (kind) {
        case kU256: k_decode_int<kU256><<<grid_for(n * 32), kBlock, 0, s>>>(plain, static_cast<u64 *>(values), n); break;
        case kFrac64: k_decode_frac<<<grid_for(n), kBlock, 0, s>>>(plain, static_cast<double *>(values), n); break;
        default: k_decode_int<kU64><<<grid_for(n * 32), kBlock, 0, s>>>(plain, static_cast<u64 *>(values), n); break;
    }
    count_launches(1);
    return cudaGetLastError();
}

}  // namespace fheb
