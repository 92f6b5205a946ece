// Compile-time parameter set of the testnet (reference: /root/reference/src/testnet.rs:8-14)
// plus the BEHZ auxiliary base SEAL 4.0 derives from it (RNSTool::initialize; restated in
// context.cpp, which re-derives these values at start-up and refuses to run on a mismatch).
#pragma once
#include <cstdint>

namespace fheb {

typedef uint64_t u64;
typedef unsigned int u32;

constexpr int kLogN = 12;
constexpr int kN = 1 << kLogN;
constexpr u64 kT = 4096;  // plain modulus
constexpr int kLogT = 12;

// modulus indices
enum : int { MQ0 = 0, MQ1 = 1, MP = 2, MB0 = 3, MB1 = 4, MSK = 5, kNumMod = 6 };

constexpr u64 kModulus[kNumMod] = {
    0xffffee001ull,          // q0  (36 bit)
    0xffffc4001ull,          // q1  (36 bit)
    0x1ffffe0001ull,         // P   (37 bit, special / key-switch prime)
    0x1ffffffffffa4001ull,   // b0  (61 bit)  BEHZ base B
    0x1ffffffffff92001ull,   // b1  (61 bit)
    0x1ffffffffffde001ull,   // m_sk (61 bit)
};
constexpr u64 kGamma = 0x1ffffffffffce001ull;  // decrypt-only aux prime
constexpr u64 kMTilde = 1ull << 32;

// The GPU's own auxiliary base for the BEHZ multiply (DESIGN.md section 4): the result of bfv_multiply is a function of integer
// polynomials that does not depend on which auxiliary primes carry them, so the tensor product runs on six primes below 2^30
// (the largest NTT primes there: 1 mod 2N), two per 64-bit word ("dual limb" d holds residues mod kDualPrime[2d] in its low
// and mod kDualPrime[2d+1] in its high 32 bits): a butterfly is one IMAD.HI + two IMAD per lane on the SM's 32-bit
// multiplier instead of 6 IMAD.WIDE + 4 IMAD for a 61-bit prime.  Product ~ 2^180 > 2 |t D| (< 2^167).
constexpr int kNumDual = 3;
constexpr u32 kDualPrime[2 * kNumDual] = {0x3fff4001u, 0x3ffee001u, 0x3ffea001u, 0x3ffe8001u, 0x3ffd6001u, 0x3ffc0001u};
// every twiddle table has kN entries in SEAL's bit-reversed order followed by a copy of entries 512..4095 regrouped for the
// transform pass that owns stages 9..11 (thread t needs entries 512+t, 1024+2t+h, 2048+4t+h): slot-major [7][512], so that a
// warp's loads are contiguous 512-byte runs instead of 32 sectors scattered over 2 KiB
constexpr int kTwPass9 = 7 * 512;
constexpr int kTwEntries = kN + kTwPass9;
constexpr int kNumTab = kNumMod + kNumDual;  // twiddle tables: the six 64-bit-lane moduli, then the three dual limbs

// floor(2^128 / q) as (hi, lo), q < 2^63 and not a power of two
struct U128c {
    u64 hi, lo;
};
constexpr U128c barrett_ratio(u64 q) {
    u64 rem = 1, hi = 0, lo = 0;
    for (int i = 0; i < 128; i++) {
        rem <<= 1;
        u64 bit = rem >= q ? 1 : 0;
        if (bit) rem -= q;
        hi = (hi << 1) | (lo >> 63);
        lo = (lo << 1) | bit;
    }
    return U128c{hi, lo};
}

}  // namespace fheb
