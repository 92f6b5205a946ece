/*
 * fhe_precompiles_b200 -- C ABI of the B200-native BFV precompile engine.
 *
 * Part 1 is the drop-in boundary: exactly the symbols the reference's staticlib exports
 * (/root/reference/src/c_fhe.rs:8-141, stamped by create_c_precompile_function! at c_fhe.rs:74-141,
 * plus fhe_free c_fhe.rs:61-64 and fhe_error c_fhe.rs:66-71), with the same signature, ownership and
 * error codes (/root/reference/src/lib.rs:14-27).  Input framing is pack.rs:119-266.
 *
 * Part 2 (fhe_b200_*) is the batch / device-resident extension the north star asks for; the single-call
 * surface of part 1 is a batch of one over the same engine.  There is no CPU fallback anywhere: without a
 * CUDA device every compute entry point fails (part 1: code 7, part 2: -1) and fhe_b200_last_error() says why.
 */
#ifndef FHE_PRECOMPILES_B200_H
#define FHE_PRECOMPILES_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- Part 1: reference surface ------------------------------------------------------------------
 * int32_t c_fhe_X(const uint8_t* bytes, size_t bytes_length, uint8_t** output, int64_t* output_length)
 *   returns 0 and a malloc'd *output (release with fhe_free) of *output_length bytes, or an error code
 *   1..7 with *output = NULL, *output_length = 0.                                  (c_fhe.rs:23-56)      */
#define FHE_PRECOMPILE(name) \
    int32_t c_fhe_##name(const uint8_t *bytes, size_t bytes_length, uint8_t **output, int64_t *output_length)

/* u256: replaces c_fhe.rs:74-84 (FheApp methods fhe.rs:161-576) */
FHE_PRECOMPILE(add_cipheru256_cipheru256);
FHE_PRECOMPILE(add_cipheru256_u256);
FHE_PRECOMPILE(add_u256_cipheru256);
FHE_PRECOMPILE(sub_cipheru256_cipheru256);
FHE_PRECOMPILE(sub_cipheru256_u256);
FHE_PRECOMPILE(sub_u256_cipheru256);
FHE_PRECOMPILE(mul_cipheru256_cipheru256);
FHE_PRECOMPILE(mul_cipheru256_u256);
FHE_PRECOMPILE(mul_u256_cipheru256);

/* u64: replaces c_fhe.rs:87-97 (FheApp methods fhe.rs:161-576) */
FHE_PRECOMPILE(add_cipheru64_cipheru64);
FHE_PRECOMPILE(add_cipheru64_u64);
FHE_PRECOMPILE(add_u64_cipheru64);
FHE_PRECOMPILE(sub_cipheru64_cipheru64);
FHE_PRECOMPILE(sub_cipheru64_u64);
FHE_PRECOMPILE(sub_u64_cipheru64);
FHE_PRECOMPILE(mul_cipheru64_cipheru64);
FHE_PRECOMPILE(mul_cipheru64_u64);
FHE_PRECOMPILE(mul_u64_cipheru64);

/* i64: replaces c_fhe.rs:100-110 (FheApp methods fhe.rs:161-576) */
FHE_PRECOMPILE(add_cipheri64_cipheri64);
FHE_PRECOMPILE(add_cipheri64_i64);
FHE_PRECOMPILE(add_i64_cipheri64);
FHE_PRECOMPILE(sub_cipheri64_cipheri64);
FHE_PRECOMPILE(sub_cipheri64_i64);
FHE_PRECOMPILE(sub_i64_cipheri64);
FHE_PRECOMPILE(mul_cipheri64_cipheri64);
FHE_PRECOMPILE(mul_cipheri64_i64);
FHE_PRECOMPILE(mul_i64_cipheri64);

/* frac64: replaces c_fhe.rs:113-123 (FheApp methods fhe.rs:161-576) */
FHE_PRECOMPILE(add_cipherfrac64_cipherfrac64);
FHE_PRECOMPILE(add_cipherfrac64_frac64);
FHE_PRECOMPILE(add_frac64_cipherfrac64);
FHE_PRECOMPILE(sub_cipherfrac64_cipherfrac64);
FHE_PRECOMPILE(sub_cipherfrac64_frac64);
FHE_PRECOMPILE(sub_frac64_cipherfrac64);
FHE_PRECOMPILE(mul_cipherfrac64_cipherfrac64);
FHE_PRECOMPILE(mul_cipherfrac64_frac64);
FHE_PRECOMPILE(mul_frac64_cipherfrac64);

/* threshold-network simulation API: replaces c_fhe.rs:126-141 (fhe.rs:594-779) */
FHE_PRECOMPILE(encrypt_u256);
FHE_PRECOMPILE(encrypt_u64);
FHE_PRECOMPILE(encrypt_i64);
FHE_PRECOMPILE(encrypt_frac64);
FHE_PRECOMPILE(reencrypt_u256);
FHE_PRECOMPILE(reencrypt_u64);
FHE_PRECOMPILE(reencrypt_i64);
FHE_PRECOMPILE(reencrypt_frac64);
FHE_PRECOMPILE(decrypt_u256);
FHE_PRECOMPILE(decrypt_u64);
FHE_PRECOMPILE(decrypt_i64);
FHE_PRECOMPILE(decrypt_frac64);
FHE_PRECOMPILE(public_key_bytes);

/* replaces c_fhe.rs:61-64: frees a buffer returned through `output` (libc free) */
void fhe_free(const uint8_t *bytes);
/* replaces c_fhe.rs:66-71: NUL-terminated message for an error code (strings of lib.rs:33-44).  The
 * reference leaks a fresh CString per call; this returns a pointer to static storage -- never free it. */
const char *fhe_error(int32_t error_code);

/* ---- Part 2: batch and device-resident extension ------------------------------------------------ */

/* Text of the last failure on the calling thread ("" if none). Valid until the thread's next call. */
const char *fhe_b200_last_error(void);
/* Number of usable CUDA devices (0 if none). */
int32_t fhe_b200_device_count(void);
/* Builds the per-device context (twiddles in HBM, constants, kernel attributes). 0 / -1. */
int32_t fhe_b200_init(int32_t device);
/* Kernels launched by this process so far (for benchmark bookkeeping). */
uint64_t fhe_b200_launch_count(void);

/* One entry of a through-the-byte-surface batch. `op` indexes fhe_b200_op_name(). */
typedef struct fhe_b200_call {
    int32_t op;            /* in : precompile index, see fhe_b200_op_index() */
    int32_t status;        /* out: 0 or lib.rs error code */
    const uint8_t *bytes;  /* in : packed input (pack.rs framing) */
    size_t bytes_length;   /* in */
    uint8_t *output;       /* out: malloc'd result, release with fhe_free */
    int64_t output_length; /* out */
} fhe_b200_call;
/* Index of a precompile by its reference name without the c_fhe_ prefix (e.g. "mul_cipheri64_cipheri64"); -1 if unknown. */
int32_t fhe_b200_op_index(const char *name);
const char *fhe_b200_op_name(int32_t index);
/* Runs n independent precompile calls, codec on `host_threads` host threads (0 = all cores), arithmetic
 * sharded over every visible GPU. Returns the number of calls whose status != 0. */
int64_t fhe_b200_batch(fhe_b200_call *calls, size_t n, int32_t host_threads);

/* Device-resident entry points. All pointers are device memory on `device`; `stream` is a cudaStream_t
 * (NULL = default stream); work is enqueued, not synchronised. Return 0 / -1.
 * Layouts (uint64 words, limb-major): ciphertext [2 polys][2 limbs q0,q1][4096]; size-3 ciphertext
 * [3][2][4096]; relin key [2 digits][2 polys][3 limbs q0,q1,P][4096] (NTT form as stored in the key file);
 * plaintext [4096] uint16 coefficients < 4096. n = number of independent ops (batch dimension outermost). */
int32_t fhe_b200_add(int32_t device, const uint64_t *a, const uint64_t *b, uint64_t *out, size_t n, void *stream);
int32_t fhe_b200_sub(int32_t device, const uint64_t *a, const uint64_t *b, uint64_t *out, size_t n, void *stream);
int32_t fhe_b200_negate(int32_t device, const uint64_t *a, uint64_t *out, size_t n, void *stream);
/* mode bit0: subtract the plaintext instead of adding; bit1: negate the result (pt - ct) */
int32_t fhe_b200_plain_addsub(int32_t device, const uint64_t *ct, const uint16_t *plain, uint64_t *out, size_t n,
                              int32_t mode, void *stream);
int32_t fhe_b200_multiply_plain(int32_t device, const uint64_t *ct, const uint16_t *plain, uint64_t *out, size_t n,
                                void *stream);
/* BFV multiply (BEHZ) without / with relinearisation */
int32_t fhe_b200_multiply(int32_t device, const uint64_t *a, const uint64_t *b, uint64_t *out3, size_t n, void *stream);
int32_t fhe_b200_relinearize(int32_t device, const uint64_t *c3, const uint64_t *rk, uint64_t *out, size_t n, void *stream);
int32_t fhe_b200_mul_relin(int32_t device, const uint64_t *a, const uint64_t *b, const uint64_t *rk, uint64_t *out,
                           size_t n, void *stream);
/* Deterministic public-key encryption of n plaintexts (uint16 [n][4096]) under pk [2][3][4096] (NTT form, as in the key
 * file) with one 512-bit seed per op (seeds [n][8] words; the byte surface passes the eight little-endian words of its
 * SHA-512 digest, fhe.rs:611-616).  BIT-EXACT with the reference: this is sunscreen 0.8.1 `encrypt_deterministic` as the
 * Sunscreen SEAL fork computes it -- Blake2xb PRNG keyed with the seed, std::uniform_int_distribution ternary u and
 * clipped std::normal_distribution errors (libstdc++, the Linux build), encryption at the data level without the special
 * modulus -- reproduced on the GPU (k_seal_prng / k_seal_sample / k_encrypt_seal) and pinned by the reference's own SHA-512
 * known answers (fhe.rs:2101-2244) through c_fhe_encrypt_u256 / c_fhe_reencrypt_u256 in the GPU tests.
 * Decryption of n size-2 ciphertexts with sk [>=2 limbs][4096] (NTT form) -> plaintexts. */
int32_t fhe_b200_encrypt(int32_t device, const uint64_t *pk, const uint16_t *plain, const uint64_t *seeds, uint64_t *ct, size_t n,
                         void *stream);
int32_t fhe_b200_decrypt(int32_t device, const uint64_t *ct, const uint64_t *sk, uint16_t *plain, size_t n, void *stream);
/* The sampling stage of fhe_b200_encrypt on its own, on caller-supplied draws instead of the Blake2xb stream: op i owns
 * fhe_b200_seal_op_words() device words at streams + i * that -- 28,672 32-bit draws (little-endian word pairs) followed by
 * room for the three int8[4096] polynomials u, e0, e1, which are written there in SEAL's order (sample_poly_ternary, then
 * sample_poly_normal twice; libstdc++ distributions).  failed[i] = 1 when the draws ran out.  Lets tests drive the rare
 * paths (a zero draw inside u, a clipped variate) that no searchable seed reaches. */
int32_t fhe_b200_seal_sample(int32_t device, uint64_t *streams, int32_t *failed, size_t n, void *stream);
size_t fhe_b200_seal_op_words(void);
/* The same with SEAL's invariant-noise-budget test: exhausted[i] (device ints) = 1 where ciphertext i has no budget left
 * (max |t x mod q| centred >= 2^70), i.e. where sunscreen's Runtime::decrypt fails and c_fhe_decrypt_* / c_fhe_reencrypt_*
 * return 5 (FailedDecryption, fhe.rs:640-643, 692-696); plain[i] is then meaningless. */
int32_t fhe_b200_decrypt_checked(int32_t device, const uint64_t *ct, const uint64_t *sk, uint16_t *plain, int32_t *exhausted, size_t n,
                                 void *stream);
/* Typed values <-> plaintexts on the device: sunscreen's encoders of the four operand kinds, so that a device-resident chain
 * can start and end in values (fhe_b200_encode_values -> fhe_b200_encrypt / plain_addsub / multiply_plain ... ->
 * fhe_b200_decrypt_checked -> fhe_b200_decode_values).  `kind` is numbered as in fhe_b200_data_type_kind: 0 u256, 1 u64, 2 i64,
 * 3 frac64.  `values` holds one value per op, batch outermost: u64 uint64; i64 int64; u256 four uint64 words, least
 * significant first; frac64 an IEEE double.  `plain` is [n][4096] uint16, 16-byte aligned (any cudaMalloc pointer).
 * BIT-EXACT with the byte surface: row i of encode equals the plaintext c_fhe_*_<kind> builds from the value's big-endian
 * serialization (Unsigned64 / Unsigned256 / Signed / Fractional<64> encoders, every one of the 4096 coefficients), and decode
 * is the same function of EVERY uint16 plaintext as c_fhe_decrypt_<kind>'s decoder, coefficients >= 4096 included (they wrap
 * as in the reference's release arithmetic); for frac64 that is the double the host's in-order sum gives, bit for bit.
 * status (device, [n], may be NULL): 0, or 7 (the byte surface's code) where a frac64 value is NaN, +-inf or |v| >= 2^64;
 * that row is all zero.  The integer kinds never fail.  Device pointers, enqueued on `stream`; n == 0 launches nothing.
 * 0 / -1 (unknown kind, misaligned plain, no device, launch failure: see fhe_b200_last_error). */
int32_t fhe_b200_encode_values(int32_t device, int32_t kind, const void *values, uint16_t *plain, int32_t *status, size_t n, void *stream);
int32_t fhe_b200_decode_values(int32_t device, int32_t kind, const uint16_t *plain, void *values, size_t n, void *stream);
/* Same op on HOST buffers (pin them for full PCIe rate): copies in, computes and copies out chunk by chunk with
 * the three phases of consecutive chunks overlapped; returns when `out` is complete. rk: host words. */
int32_t fhe_b200_mul_relin_host(int32_t device, const uint64_t *a, const uint64_t *b, const uint64_t *rk, uint64_t *out,
                                size_t n);
/* Same op on SERIALIZED operands. Operand i of an array is the zstd frame at frames + i * stride: the compressed body of a
 * ciphertext as this library serializes it (a "structured frame": fhe_b200_frame_bytes() = 82,054 bytes, at byte 148 of the
 * packed `Ciphertext`; what every precompile here returns and what chained calls carry). Frames cross PCIe as they are (5 bytes
 * per residue instead of 8), are validated and unpacked on the GPU, and result i is written as a frame at
 * out_frames + i * fhe_b200_frame_stride(). Pin the buffers for full PCIe rate. status[i]: 0 done; 1 an operand is not a
 * structured frame or fails SEAL's range checks (result undefined: send that call through c_fhe_mul_*); 2 the result is not
 * representable as a structured frame (transparent ciphertext). Replaces, for a batch, the bincode + SEAL load/save around
 * Evaluator::multiply + relinearize_inplace in fhe_binary_op (/root/reference/src/fhe.rs:21-30). */
int32_t fhe_b200_mul_relin_frames(int32_t device, const uint8_t *a_frames, const uint8_t *b_frames, size_t stride, const uint64_t *rk,
                                  uint8_t *out_frames, size_t n, int32_t *status);
/* Device-resident ciphertexts from / to SERIALIZED form, so that a chain of device-resident operations (fhe_b200_add ...
 * fhe_b200_mul_relin on device pointers) crosses PCIe once at each end instead of once per operation.
 * upload: n structured frames (host, `stride` apart, as for fhe_b200_mul_relin_frames) -> d_words [n][2][2][4096] on `device`,
 *   validated like SEAL's checked load; status[i] (host, may be NULL): 0 ok, 1 not a structured frame or a residue >= q.
 * download: d_words -> n structured frames at out_frames + i * fhe_b200_frame_stride() (host); status[i]: 0 ok, 2 the
 *   ciphertext is constant (transparent) and has no structured frame (serialise it with fhe_b200_write_ciphertext).
 * Both are synchronous and pipeline chunks of 256 ciphertexts over two streams; pin the host buffers for full PCIe rate.
 * Replaces bincode::deserialize / serialize of a Ciphertext around a sequence of Runtime::run calls (fhe.rs:21-30). */
int32_t fhe_b200_upload_frames(int32_t device, const uint8_t *frames, size_t stride, size_t n, uint64_t *d_words, int32_t *status);
int32_t fhe_b200_download_frames(int32_t device, const uint64_t *d_words, size_t n, uint8_t *out_frames, int32_t *status);
size_t fhe_b200_frame_bytes(void);
size_t fhe_b200_frame_stride(void);
/* Integer-pipe peak of `device` in 1e12 multiply-adds/s, measured by a register-only microbenchmark
 * (wide: 0 mad.lo.u32 [IMAD], 1 mul.wide.u32 [IMAD.WIDE], 2 add.cc+addc, 3 mad.lo+add, 4 mul.wide+add). Denominator of the integer roofline; synchronous. */
int32_t fhe_b200_int_peak(int32_t device, int32_t wide, double *tera_mads_per_s);
/* Register-only NTT butterfly rate of `device` in 1e9 butterflies/s for modulus class of `mod` (0-2: 36/37-bit,
 * 3-5: 61-bit): the compute ceiling of the transform's inner loop without memory or barriers. */
int32_t fhe_b200_bfly_peak(int32_t device, int32_t mod, double *giga_bfly_per_s);
/* Which of the four operand kinds a Ciphertext data_type string ("<type name>,<version>,<is_encrypted>") belongs to:
 * 0 u256, 1 u64, 2 i64, 3 frac64, -1 none.  This is the check every binary precompile applies to its ciphertext operands
 * (a mismatch is code 7, like sunscreen's argument check behind fhe.rs:28).  Host only. */
int32_t fhe_b200_data_type_kind(const char *data_type);
/* Ops per chunk of the device-resident entry points (default 4,096, FHE_B200_CHUNK_OPS): a batch larger than this runs chunk
 * after chunk through one scratch arena.  ops <= 0 only queries.  Returns the previous value (-1 without a device). */
int64_t fhe_b200_set_chunk_ops(int64_t ops);
/* Per-kernel timing of fhe_b200_mul_relin (CUDA events around each launch, on the caller's stream).
 * ms / launches are indexed 1 k_floor_sk_d, 3 k_relin_finish, 4 k_ext_ntt_d, 5 k_tensor_intt_d, 6 k_digit_ntt, 7 k_ks_intt,
 * 8 k_ext_conv_d, 10 k_rk_*_ksd (key preparation), 11 k_digit_ntt_ksd, 14 k_tensor_floor_d, 15 k_ks_tail_ksd; slots 0, 2, 9,
 * 12 and 13 are reserved and stay zero.  The report synchronises the device and resets the accumulators. */
/* Phase timing of the byte surface (SURVEY 8d: parse+inflate / H2D / kernels / D2H / deflate).  When on, every binary
 * precompile call records, for the calling thread: us[0] framing + key lookup, us[1] operand decode (bincode + zstd inflate
 * + range checks), us[2] H2D, us[3] kernels, us[4] D2H (CUDA events on the lane's stream), us[5] result encode, us[6] total. */
void fhe_b200_set_call_timing(int32_t on);
void fhe_b200_last_call_breakdown(double us[7]);
void fhe_b200_set_kernel_timing(int32_t on);
int32_t fhe_b200_kernel_timing_report(int32_t device, double ms[16], uint64_t launches[16]);
/* Batched negacyclic NTT in place over n_limbs limbs of 4096 words; limb i uses modulus mods[i % n_mods]
 * (0 q0, 1 q1, 2 P, 3 b0, 4 b1, 5 m_sk). inverse != 0: bit-reversed -> natural, scaled by N^-1. */
int32_t fhe_b200_ntt(int32_t device, uint64_t *data, size_t n_limbs, const int32_t *mods, int32_t n_mods, int32_t inverse,
                     void *stream);

/* Host-side format helpers (no GPU needed): parse a sunscreen PublicKey and write its relinearisation key
 * (2*2*3*4096 words) and/or public key (2*3*4096 words); either pointer may be NULL. lib.rs error code. */
int32_t fhe_b200_parse_public_key(const uint8_t *bytes, size_t len, uint64_t *pk_words, uint64_t *rk_words);
int32_t fhe_b200_parse_private_key(const uint8_t *bytes, size_t len, uint64_t *sk_words);
/* sunscreen::Ciphertext bytes <-> 2*2*4096 coefficient words (data_type kept in a caller buffer) */
int32_t fhe_b200_parse_ciphertext(const uint8_t *bytes, size_t len, uint64_t *words, char *data_type, size_t data_type_cap);
int32_t fhe_b200_write_ciphertext(const uint64_t *words, const char *data_type, uint8_t **output, int64_t *output_length);
/* parms_id (4 words) of the key level (which = 0) or the data level (which = 1) */
/* How zstd-mode ciphertext payloads are WRITTEN: 0 (default) = libzstd level 3, byte for byte what SEAL's save() writes
 * (~88.5 KB, ~1 ms on a host core; pinned by the reference's known answers, which hash the compressed bytes);
 * 1 = structure-aware standard zstd frames laid out directly (raw 5-byte literals + repeat-offset matches for the three zero
 * bytes of every 36-bit residue; ~82 KB, memcpy speed, written on the GPU in batches) for deployments where every consumer
 * only needs a valid frame, not SEAL's exact bytes.  Both are RFC 8878 frames any SEAL build reads.  mode < 0 only queries.
 * Returns the previous mode.  Also settable with FHE_B200_ZSTD_WRITER=structured. */
/* The SHA-512 behind the encrypt / reencrypt seed (fhe.rs:600-612): portable != 0 forces the built-in implementation,
 * 0 uses libcrypto's when the machine has it.  Exposed so that tests can pin both against a known-good SHA-512. */
void fhe_b200_sha512(const uint8_t *bytes, size_t len, int32_t portable, uint8_t out[64]);
int32_t fhe_b200_set_zstd_writer(int32_t mode);
/* Device-side zstd inflate of n ciphertext-payload frames (codec_kernels.cu: k_zd2_parse, k_zd3_huf, k_zd3_seq, k_zd3_exec):
 * what fhe_b200_batch uses for the operands of a tile.  frames[i] / lens[i] are host buffers; `out` receives n payloads of
 * 131,169 bytes; status[i] = 1 when the frame was inflated (byte-identical to libzstd), 2 when the strict decoder hands it
 * back to the host (unsupported feature, malformed frame, or content that is not a 131,169-byte payload).  The batch surface
 * additionally checks the 97-byte prefix and every residue (k_ct_unpack); this entry point stops at the payload bytes.
 * elapsed_ms: kernels only. */
int32_t fhe_b200_zstd_inflate(int32_t device, const uint8_t *const *frames, const size_t *lens, size_t n, uint8_t *out,
                              int32_t *status, float *elapsed_ms);
void fhe_b200_parms_id(int32_t which, uint64_t out[4]);

#ifdef __cplusplus
}
#endif
#endif
