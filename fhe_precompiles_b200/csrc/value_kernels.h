// Launchers of the typed-value encoders and decoders (value_kernels.cu): sunscreen's plaintext encodings of Unsigned256,
// Unsigned64, Signed and Fractional<64> on the GPU, bit-identical to encode_scalar / decode_scalar (codec.cpp).
// Plain C++ header: included by c_api.cpp (g++) and nvcc.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

namespace fheb {

// Kind numbering of fhe_b200_data_type_kind (codec.h Kind): 0 u256, 1 u64, 2 i64, 3 frac64.
// values: one per op, batch outermost -- u64 / i64: one 64-bit word; u256: four words, least significant first;
// frac64: an IEEE double.  plain: [n][4096] uint16, 16-byte aligned.
bool value_kind_valid(int kind);
// status (optional, [n] on the device): 0, or 7 where encode_scalar fails (frac64 NaN, +-inf, |v| >= 2^64); such rows are zero
cudaError_t launch_encode_values(int kind, const void *values, uint16_t *plain, int32_t *status, size_t n, cudaStream_t s);
// the same function of every uint16 plaintext as decode_scalar, coefficients >= t included
cudaError_t launch_decode_values(int kind, const uint16_t *plain, void *values, size_t n, cudaStream_t s);

}  // namespace fheb
