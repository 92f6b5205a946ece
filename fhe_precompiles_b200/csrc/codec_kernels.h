// Launchers of the device-side codec (codec_kernels.cu).  Plain C++ header: included by engine.cpp (g++) and nvcc.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

namespace fheb {

constexpr int kCodecCtWords = 16384;                        // [2 polys][2 limbs][4096]
constexpr size_t kCtPrefixBytes = 97;                        // SEAL ciphertext payload bytes before the words
constexpr size_t kCtPayloadBytes = kCtPrefixBytes + 8 * 16384;  // 131,169
constexpr size_t kPayloadStride = 131200;                    // per-job payload slot on the device (8-byte aligned, slack for word loads)
constexpr size_t kPackedFrameBytes = 9 + (3 + 2 + 110 + 7) + (3 + 3 + 5 * 16382 + 2 + 5);  // 82,054: the structured frame
constexpr size_t kPackedFrameStride = 82064;
constexpr size_t kFramePad = 16;                             // readable bytes required around every staged frame (zstd_dec.h kPad)
constexpr size_t kFrameSlotBytes = 139264;                   // staging slot per operand: frame <= slot - 2 pads (zstd never expands by more)

enum : int32_t { kJobNone = 0, kJobZstd = 1, kJobPacked = 2, kJobPayload = 3 };  // CodecJob::kind (3: payload inflated by the host)
enum : int32_t { kJobPending = 0, kJobOk = 1, kJobFallback = 2 };  // status

struct CodecJob {
    uint64_t src_off;  // byte offset of the frame in the staged frame buffer
    uint32_t src_len;
    int32_t kind;
    int32_t slot;     // destination ciphertext slot
    int32_t operand;  // 0: first operand array, 1: second
};

size_t codec_work_bytes();  // decoder workspace per job
// inflate + validate + unpack every job into dst_a / dst_b slots; status[j] = kJobOk or kJobFallback
// `phase`: kCodecAll, or the two halves separately - kCodecDecode (clear status[], run the zstd decoder) and kCodecUnpack
// (validate + unpack payloads and structured frames) - so that a tile can inflate part of its frames on the host between them
enum : int { kCodecAll = 0, kCodecDecode = 1, kCodecUnpack = 2 };
cudaError_t launch_codec_inflate(const uint8_t *frames, uint8_t *payloads, const CodecJob *jobs, int32_t *status, void *work,
                                 const uint8_t *prefix, uint64_t *dst_a, uint64_t *dst_b, int n_jobs, bool any_zstd,
                                 bool any_packed, bool any_payload, cudaStream_t s, int phase = kCodecAll);
// n result ciphertexts -> n structured frames (kPackedFrameStride apart); constant_flag[i] = 1 if the host must use libzstd instead
cudaError_t launch_codec_pack(const uint64_t *words, uint8_t *frames, int32_t *constant_flag, const uint8_t *prefix, int n,
                              cudaStream_t s);
uint64_t codec_launch_count();

}  // namespace fheb
