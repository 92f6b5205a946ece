// Launchers of the sm_100a kernels in kernels.cu (device pointers, caller-chosen stream).
#pragma once
#include <cstddef>

#include "devconsts.h"

namespace fheb {

struct LimbMods {
    int n;               // limbs per polynomial in the caller's layout
    int mod[kNumMod];    // modulus index of each limb
};

cudaError_t upload_constants(const DevConsts &c, const DevTables &t, const DevTwLow &lo);  // to the current device
cudaError_t kernels_configure();                                       // opt-in shared memory sizes, current device

// data: n_limbs consecutive 4096-word limbs, limb i uses modulus mods.mod[i % mods.n]; in place
cudaError_t launch_ntt(u64 *data, size_t n_limbs, const LimbMods &mods, bool inverse, cudaStream_t s);
// op: 0 add, 1 sub, 2 negate(a)
cudaError_t launch_eltwise(const u64 *a, const u64 *b, u64 *out, size_t n_ops, int op, cudaStream_t s);
// mode bit0: subtract, bit1: negate result
cudaError_t launch_plain_addsub(const u64 *ct, const unsigned short *plain, u64 *out, size_t n_ops, int mode, cudaStream_t s);
cudaError_t launch_mul_plain(const u64 *ct, const unsigned short *plain, u64 *out, size_t n_ops, cudaStream_t s);
// BEHZ multiply on the dual base; scratch: nttbuf [n][4][5][N], tens [n][3][5][N]
cudaError_t launch_ext_conv(const u64 *a, const u64 *b, u64 *nttbuf, size_t n_ops, cudaStream_t s);
cudaError_t launch_ext_ntt(u64 *nttbuf, size_t n_ops, cudaStream_t s);  // in place, after launch_ext_conv
// then either launch_tensor_intt + launch_floor_sk, or both in one kernel (launch_tensor_floor) -> c3 [n][3][2][N]
cudaError_t launch_tensor_intt(const u64 *nttbuf, u64 *tens, size_t n_ops, cudaStream_t s);
cudaError_t launch_floor_sk(const u64 *tens, u64 *c3, size_t n_ops, cudaStream_t s);
cudaError_t launch_tensor_floor(const u64 *nttbuf, u64 *c3, size_t n_ops, cudaStream_t s);
// key switch on SEAL's key primes: launch_digit_ntt -> launch_ks_intt -> launch_relin_finish; dig, ks [n][2][3][N]
cudaError_t launch_digit_ntt(const u64 *c3, u64 *dig, size_t n_ops, cudaStream_t s);
cudaError_t launch_ks_intt(const u64 *dig, const u64 *rk, u64 *ks, size_t n_ops, cudaStream_t s);
// the same with a key per op: key_index [n_ops] device ints, op i under the key rks[key_index[i]] (rks: device array of device
// pointers to keys [2][2][3][N]; indices not checked).  key_index null: every op under rk, as launch_ks_intt.
cudaError_t launch_ks_intt_keyed(const u64 *dig, const u64 *rk, const u64 *const *rks, const int *key_index, u64 *ks, size_t n_ops,
                                 cudaStream_t s);
cudaError_t launch_relin_finish(const u64 *c3, const u64 *ks, u64 *out, size_t n_ops, cudaStream_t s);
// decrypt n size-2 ciphertexts with sk [>=2 limbs][N] (NTT form): xbuf scratch [n][2][N], plain out [n][N] u16
// exhausted (optional, [n_ops] ints on the device): set to 1 where the invariant noise budget is 0
cudaError_t launch_decrypt(const u64 *ct, const u64 *sk, u64 *xbuf, unsigned short *plain, size_t n_ops, cudaStream_t s,
                           int *exhausted = nullptr);
// deterministic pk-encryption of n plaintexts under pk [2][3][N] (NTT form), bit-exact with the reference's
// encrypt_deterministic for the per-op 512-bit seeds; encbuf: scratch [n][6][N] words (PRNG stream + samples);
// failed[op] (optional) = 1 if the op's PRNG stream window ran out (never observed: ~24 sigma)
cudaError_t launch_encrypt(const u64 *pk, const unsigned short *plain, const u64 *seeds, u64 *encbuf, u64 *ct, size_t n_ops,
                           cudaStream_t s, int *failed = nullptr);
// the same with a key per op: pks [k][2][3][N], key_index [n_ops] device ints in [0, k) (not checked: an index outside the
// key array is the caller's error, as a bad pointer is); op i encrypts under pks + key_index[i] * 2 * 3 * N
cudaError_t launch_encrypt_keyed(const u64 *pks, const int *key_index, const unsigned short *plain, const u64 *seeds, u64 *encbuf,
                                 u64 *ct, size_t n_ops, cudaStream_t s, int *failed = nullptr);
// SEAL's samplers (ternary u, clipped-normal e0 / e1) on caller-supplied streams of 32-bit draws: op i owns
// kSealOpWords = 28 * 512 + 3 * N / 8 words at streams + i * kSealOpWords -- 28,672 draws followed by room for the three
// int8 sample polynomials, which the kernel writes there.  failed[i] = 1 if the draws ran out.
constexpr size_t kSealOpWords = 28 * 512 + 3 * 4096 / 8;
cudaError_t launch_seal_sample(u64 *streams, signed char *samples, int *failed, size_t n_ops, cudaStream_t s);
// key switch on the dual base: launch_rk_prepare_ksd (per chunk) -> launch_digit_ntt_ksd -> launch_ks_tail_ksd
// tmp36: 36 limbs of scratch; the dual-NTT key ends up at tmp36 + 24 limbs
cudaError_t launch_rk_prepare_ksd(const u64 *rk, u64 *tmp36, cudaStream_t s);
// K keys in the same three launches: the keys rks[0 .. K) (a device array of device pointers), or rk itself when rks is null
// (K = 1); tmp: 24 K limbs of scratch; rkd: the prepared keys [K][12][N].  K <= kMaxPrepareKeys.
constexpr size_t kMaxPrepareKeys = 65535;
cudaError_t launch_rk_prepare_keys(const u64 *rk, const u64 *const *rks, size_t n_keys, u64 *tmp, u64 *rkd, cudaStream_t s);
cudaError_t launch_digit_ntt_ksd(const u64 *c3, u64 *dig, size_t n_ops, cudaStream_t s);
// key_index (optional, [n_ops] device ints, not checked): op i under the prepared key rkd + key_index[i] * 12 * N
cudaError_t launch_ks_tail_ksd(const u64 *dig, const u64 *rkd, const u64 *c3, u64 *out, size_t n_ops, cudaStream_t s,
                               const int *key_index = nullptr);
// table[i] = rks + i * stride for i < n_keys (device memory): the key table of contiguous keys
cudaError_t launch_key_table(const u64 *rks, size_t stride, size_t n_keys, const u64 **table, cudaStream_t s);

uint64_t launch_count();
void count_launches(uint64_t n);  // kernels replayed through a CUDA graph (the launchers only count at capture time)
// integer multiply-add peak of the current device in 1e12 mad/s (microbenchmark, synchronous)
cudaError_t measure_int_peak(int mode, double *tera_ops_per_s);
// register-only NTT butterfly rate (1e9 butterflies/s) for a small (mod < 3) or a 61-bit prime
cudaError_t measure_bfly_peak(int mod, double *giga_bfly_per_s);

}  // namespace fheb
