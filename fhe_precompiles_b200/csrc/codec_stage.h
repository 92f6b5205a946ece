// Staging of serialized ciphertext operands for launch_codec_inflate: which libzstd frames the GPU inflates, and where each
// job's frame or payload sits in the pinned staging.  The byte surface's tiles and single calls and Engine::upload_ciphertexts
// all lay out their jobs here.  Host only; it needs nothing beyond codec_kernels.h, so a test builds it with g++ alone.
#pragma once
#include <cstddef>
#include <cstdint>

#include "codec_kernels.h"

namespace fheb {

// how one ciphertext operand reaches the device words (classified by engine.cpp from its bincode framing and SEAL header)
enum class Route : uint8_t {
    Reject,  // the bincode framing fails: its code is the result
    Host,    // decode_ciphertext decides: wrong data_type, malformed SEAL header or a zstd frame too large for a staging slot
    Blob,    // compr_mode none or zlib: the host inflates the blob into a payload slot
    Zstd,    // a libzstd-written frame
    Packed,  // a structured frame (always kPackedFrameBytes)
};

// libzstd-written operand frames of a tile (or transfer chunk) are inflated on the GPU when it brings at least this many of
// them, else on the host: a frame is a 16 k-step chain, ~3 ms on the GPU however few frames there are, 0.11 ms on a host core
constexpr size_t kDeviceZstdMinFrames = 128;
inline bool device_inflates(size_t lib_frames) { return lib_frames >= kDeviceZstdMinFrames; }

struct StageOperand {
    Route route;
    size_t frame_len;        // Zstd, Packed: length of the zstd frame (it fits a kFrameSlotBytes slot with both pads)
    int32_t slot, operand;   // CodecJob::slot / operand: where launch_codec_inflate writes the words
};

struct StagePlan {
    int jobs = 0;
    int payloads = 0;        // P: jobs [0, P) carry payloads the host inflates, job j's at payloads + j * kPayloadStride
    size_t frame_bytes = 0;  // the frames the device reads fill [0, frame_bytes) of the frame staging
    bool any_zstd = false, any_packed = false;
};

// Jobs for ops[0, n) into jobs[] (room for n): one payload job per Blob, and per Zstd unless device_inflates(the number of
// Zstd operands), in operand order; then one job per frame the device reads, at a 16-byte aligned offset with kFramePad
// readable bytes on either side.  job[i] = the job of operand i, or -1 for Reject and Host.  The layout depends on the routes
// and the lengths of the frames the device reads only: a single call (its libzstd frames always inflated on the host) has one
// layout per pair of routes.
inline StagePlan plan_codec_jobs(const StageOperand *ops, size_t n, CodecJob *jobs, int32_t *job) {
    size_t lib_frames = 0;
    for (size_t i = 0; i < n; i++) lib_frames += ops[i].route == Route::Zstd;
    const bool dev_zstd = device_inflates(lib_frames);
    StagePlan p;
    for (size_t i = 0; i < n; i++) {
        const StageOperand &o = ops[i];
        job[i] = -1;
        if (o.route != Route::Blob && !(o.route == Route::Zstd && !dev_zstd)) continue;
        job[i] = p.jobs;
        jobs[p.jobs++] = CodecJob{0, 0, kJobPayload, o.slot, o.operand};
    }
    p.payloads = p.jobs;
    for (size_t i = 0; i < n; i++) {
        const StageOperand &o = ops[i];
        if (o.route != Route::Packed && !(o.route == Route::Zstd && dev_zstd)) continue;
        job[i] = p.jobs;
        jobs[p.jobs++] = CodecJob{p.frame_bytes + kFramePad, (uint32_t)o.frame_len, o.route == Route::Packed ? kJobPacked : kJobZstd,
                                  o.slot, o.operand};
        (o.route == Route::Packed ? p.any_packed : p.any_zstd) = true;
        p.frame_bytes += (o.frame_len + 2 * kFramePad + 15) & ~(size_t)15;
    }
    return p;
}

}  // namespace fheb
