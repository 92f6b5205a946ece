// Byte-level formats of the precompile surface, host side.
//   outer framing ............ /root/reference/src/pack.rs:119-266 (BE u32 offsets)
//   scalar operands .......... /root/reference/src/pack.rs:47-104 (BE bytes)
//   Ciphertext / PublicKey ... bincode 1.3.3 (Cargo.toml:10) over sunscreen 0.8.1 serde types wrapping
//                              SEAL 4.0 save() streams (zstd / zlib / none); layouts in SURVEY.md App. A,
//                              established from the reference's key fixtures.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "params.h"

namespace fheb {

// error codes of /root/reference/src/lib.rs:14-27
enum : int32_t {
    kOk = 0,
    kErrUnexpectedEOF = 1,
    kErrPlatformArchitecture = 2,
    kErrInvalidEncoding = 3,
    kErrOverflow = 4,
    kErrFailedDecryption = 5,
    kErrFailedEncryption = 6,
    kErrSunscreen = 7,
};

struct Span {
    const uint8_t *p = nullptr;
    size_t n = 0;
};

// pack.rs:238-266 with bounds checks (the reference panics on out-of-range offsets; we return 1)
int32_t unpack_binary_operation(Span in, Span *pk, Span *a, Span *b);
// pack.rs:153-175
int32_t unpack_two_arguments(Span in, Span *a, Span *b);

constexpr size_t kParamsBytes = 56;  // sunscreen Params for 3 coefficient primes: N,k,3 primes,t (u64) + scheme,security (u32)
constexpr size_t kCtHeaderBytes = 97;  // SEAL ciphertext payload bytes before the coefficient words
constexpr size_t kCtWords = 2 * 2 * kN;

// Decoded view of a sunscreen::Ciphertext holding one data-level, size-2, coefficient-form SEAL ciphertext.
struct CipherView {
    std::string data_type;          // opaque "<type>,<version>,<is_encrypted>"
    uint8_t params[kParamsBytes];   // WithContext params, echoed into the result
    uint8_t compr_mode = 2;         // SEAL compr_mode of the blob, echoed into the result
};

// Parses `in`, validates it like SEAL's checked load (parms_id, sizes, coefficient ranges) and writes the
// 16384 coefficient words to `words` (caller-owned, e.g. pinned staging).  Returns an lib.rs error code.
int32_t decode_ciphertext(Span in, CipherView *view, uint64_t *words);

// The pieces of decode_ciphertext / encode_ciphertext the device codec path needs (engine.cpp, codec_kernels.cu):
// bincode framing only (data_type, params checks; `blob` = the SEAL blob inside)
int32_t parse_ciphertext_framing(Span in, CipherView *view, Span *blob);
// SEAL header of the blob: -1 malformed, 0 not zstd (compr none / zlib: host path), 1 zstd frame, 2 zstd frame in this library's
// structured layout (every header byte verified); `frame` = the zstd frame, `compr` = the blob's compr_mode
int classify_ciphertext_blob(Span blob, Span *frame, uint8_t *compr);
// libzstd inflate of a ciphertext frame straight into `dst` (131,169 bytes, e.g. pinned staging); false unless the frame
// holds exactly a payload of that size.  The content is validated on the device (k_ct_unpack).
bool inflate_ct_payload(Span frame, uint8_t *dst);
// the same for a whole SEAL blob of any compr_mode (none: copied, zlib, zstd); false unless it holds exactly such a payload
bool inflate_ct_blob(Span blob, uint8_t *dst);
// the 97 bytes every valid size-2 data-level coefficient-form ciphertext payload starts with
void canonical_ct_prefix(uint8_t *prefix97);
// bincode(Ciphertext) around an already compressed payload `body` (SEAL header with view.compr_mode added here)
void wrap_ciphertext_blob(const CipherView &view, const uint8_t *body, size_t body_len, std::vector<uint8_t> *out);
// the same into a caller-provided buffer of wrapped_ciphertext_size(view, body_len) bytes
size_t wrapped_ciphertext_size(const CipherView &view, size_t body_len);
void wrap_ciphertext_blob_to(const CipherView &view, const uint8_t *body, size_t body_len, uint8_t *dst);

// Serialises a size-2 data-level ciphertext (bincode + SEAL + compression) into `out`.
int32_t encode_ciphertext(const CipherView &view, const uint64_t *words, std::vector<uint8_t> *out);
// zstd writer for ciphertext payloads: 1 (default) = structure-aware standard frames (codec.cpp), 0 = libzstd level 3
void set_zstd_writer(int mode);
int zstd_writer();

// Parses a sunscreen::PublicKey; if `rk_words` is non-null the relinearisation key is written there as
// [digit 0..1][poly 0..1][limb q0,q1,P][N] (2*2*3*4096 words).  `has_relin` reports whether the key
// carries relin keys.  Returns an lib.rs error code.
constexpr size_t kRkWords = 2 * 2 * 3 * kN;
constexpr size_t kPkWords = 2 * 3 * kN;
int32_t decode_public_key(Span in, uint64_t *pk_words, uint64_t *rk_words, bool *has_relin);
// Parses a sunscreen::PrivateKey into [limb q0,q1,P][N] (NTT form)
int32_t decode_private_key(Span in, uint64_t *sk_words);

// scalar operands (pack.rs:47-104) -> plaintext polynomial (sunscreen encoders, SURVEY App. D)
enum class Kind : int { U256 = 0, U64 = 1, I64 = 2, Frac64 = 3 };
// plain: kN u16 coefficients, zero padded.  Returns lib.rs error code (3 for a wrong byte length,
// 7 when sunscreen's encoder would reject the value, e.g. NaN).
int32_t encode_scalar(Kind kind, Span bytes, uint16_t *plain);
// plaintext polynomial -> big-endian scalar bytes
void decode_scalar(Kind kind, const uint16_t *plain, size_t len, std::vector<uint8_t> *out);
// the `Ciphertext.data_type` string sunscreen 0.8.1 writes for an encrypted value of `kind`, and the argument check against it
const char *data_type_of(Kind kind);
bool data_type_matches(const std::string &data_type, Kind kind);

// zstd is loaded from libzstd.so.1 at first use (no headers in the image); throws if missing
bool zstd_available();

}  // namespace fheb
