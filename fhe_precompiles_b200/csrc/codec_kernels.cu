// Device side of the byte surface (SURVEY 8f-3): the zstd frames of the ciphertext operands are inflated on the GPU and the
// result is written as a structured zstd frame on the GPU, so the host moves compressed bytes only.
//   k_zd2_parse    : headers and FSE / Huffman tables, thread per frame (zstd_plan2.h)
//   k_zd3_huf      : Huffman literal streams, thread per stream (zstd_plan2.h)
//   k_zd3_seq      : FSE sequence chains, four frames per warp, tables in shared memory (zstd_plan2.h, zstd_plan3.cuh)
//   k_zd3_exec     : sequence execution, CTA per frame (zstd_plan3.cuh, zstd_exec3.h)
//   k_ct_unpack    : 131,169-byte SEAL payload -> [2][2][N] words; checks the 97-byte prefix against the only value a valid
//                    data-level ciphertext can have and every residue against its modulus
//   k_unpack40     : the same for frames in this library's own structured layout (5-byte literals), fully parallel
//   k_ct_pack40    : [2][2][N] words -> the complete structured frame (codec.cpp zstd_pack40 layout), byte for byte
// Anything unusual is flagged and the host redoes that call with libzstd (codec.cpp), whose verdict is authoritative.
#include <atomic>

#include "codec_kernels.h"
#include "params.h"
#include "zstd_plan3.cuh"

namespace fheb {

extern std::atomic<unsigned long long> g_codec_launches;
std::atomic<unsigned long long> g_codec_launches{0};

namespace {
constexpr u64 kQ0 = kModulus[0], kQ1 = kModulus[1];

struct JobScratch {  // one workspace slot per job, shared by the four inflate kernels
    zd::Plan2 plan;
    zd::Work work;  // table-construction scratch of the parse step
    zd::Tables2 tabs;
    uint64_t seqs[zd::kP2MaxSeqs];
    uint8_t lits[(kCtPayloadBytes + 16 + 7) & ~(size_t)7];
};

__global__ void __launch_bounds__(32) k_zd2_parse(const uint8_t *frames, const CodecJob *jobs, JobScratch *scratch, int n) {
    const int j = blockIdx.x * 32 + threadIdx.x;
    if (j >= n) return;
    const CodecJob job = jobs[j];
    JobScratch *sc = &scratch[j];
    sc->plan.status = zd::kZdFallback;
    if (job.kind != kJobZstd) return;
    zd::work_bind(&sc->work, nullptr);
    zd::plan2_parse(frames + job.src_off, job.src_len, kCtPayloadBytes, &sc->work, &sc->plan, &sc->tabs);
}
__global__ void __launch_bounds__(128) k_zd3_huf(const uint8_t *frames, const CodecJob *jobs, JobScratch *scratch, int n) {
    const int j = blockIdx.x * 32 + (threadIdx.x & 31), role = threadIdx.x >> 5;
    if (j >= n) return;
    const CodecJob job = jobs[j];
    if (job.kind != kJobZstd) return;
    JobScratch *sc = &scratch[j];
    sc->plan.huf_bad[role] = zd::plan2_huf(frames + job.src_off, &sc->plan, &sc->tabs, sc->lits, role) ? 0 : 1;
}
__global__ void __launch_bounds__(32) k_zd3_seq(const uint8_t *frames, const CodecJob *jobs, JobScratch *scratch, int n) {
    extern __shared__ __align__(16) uint8_t smem3[];
    const int j = blockIdx.x * zd3::kSeqFrames + (threadIdx.x >> 3);
    const bool in_range = j < n;
    const CodecJob job = in_range ? jobs[j] : CodecJob{0, 0, kJobNone, 0, 0};
    JobScratch *sc = &scratch[in_range ? j : 0];
    const bool have = in_range && job.kind == kJobZstd && sc->plan.status == zd::kZdOk;
    const bool ok = zd3::seq_frames(frames + job.src_off, &sc->plan, &sc->tabs, sc->seqs, have, (uint32_t *)smem3);
    if (have && (threadIdx.x & 7) == 0) sc->plan.seq_bad = ok ? 0 : 1;
}
__global__ void __launch_bounds__(zd3::kExecThreads, 1) k_zd3_exec(const uint8_t *frames, uint8_t *payloads, const CodecJob *jobs,
                                                                     int32_t *status, JobScratch *scratch, int n) {
    extern __shared__ __align__(16) uint8_t smem3[];
    for (int j = blockIdx.x; j < n; j += gridDim.x) {
        const CodecJob job = jobs[j];
        if (job.kind != kJobZstd) continue;
        JobScratch *sc = &scratch[j];
        const zd::Plan2 *plan = &sc->plan;
        int rc = zd::kZdFallback;
        if (plan->status == zd::kZdOk && !plan->seq_bad && !plan->huf_bad[0] && !plan->huf_bad[1] && !plan->huf_bad[2] && !plan->huf_bad[3] &&
            plan->content == kCtPayloadBytes)
            rc = zd3::exec_frame(frames + job.src_off, plan, sc->seqs, sc->lits, payloads + (size_t)j * kPayloadStride, smem3);
        __syncthreads();  // the shared buffers are reused by the next frame
        if (threadIdx.x == 0) status[j] = rc == zd::kZdOk ? kJobOk : kJobFallback;
    }
}

constexpr int kSplit = 8;  // blocks per ciphertext in the parallel kernels (latency of a single call)
constexpr int kWordsPerBlock = kCodecCtWords / kSplit;

// payload (prefix 97 + 16384 words at byte offset 97) -> aligned words.  kSplit blocks of 256 threads per job.
// status protocol of the parallel kernels: the host clears status[] before the launch; a block only ever writes kJobFallback.
__global__ void __launch_bounds__(256) k_ct_unpack(const uint8_t *payloads, const CodecJob *jobs, int32_t *status, const uint8_t *prefix,
                                                   u64 *dst_a, u64 *dst_b) {
    const int j = blockIdx.x;
    const CodecJob job = jobs[j];
    if (job.kind == kJobZstd ? status[j] != kJobOk : job.kind != kJobPayload) return;
    const uint8_t *p = payloads + (size_t)j * kPayloadStride;  // 8-byte aligned
    __shared__ int bad;
    if (threadIdx.x == 0) bad = 0;
    __syncthreads();
    int mybad = 0;
    if (blockIdx.y == 0 && threadIdx.x < kCtPrefixBytes) {
        // byte 77 is SEAL's minor version inside the inner DynArray header: not constrained by the host parser either
        if (threadIdx.x != 77 && p[threadIdx.x] != prefix[threadIdx.x]) mybad = 1;
    }
    u64 *dst = (job.operand ? dst_b : dst_a) + (size_t)job.slot * kCodecCtWords;
    const u64 *p64 = (const u64 *)p;  // word i lives at bytes 97 + 8 i = 8 (12 + i) + 1
    const int lo = blockIdx.y * kWordsPerBlock;
    for (int i = lo + threadIdx.x; i < lo + kWordsPerBlock; i += 256) {
        const u64 w = (p64[12 + i] >> 8) | (p64[13 + i] << 56);
        const u64 q = ((i >> 12) & 1) ? kQ1 : kQ0;
        if (w >= q) mybad = 1;
        dst[i] = w;
    }
    if (mybad) atomicOr(&bad, 1);
    __syncthreads();
    if (threadIdx.x == 0 && bad) status[j] = kJobFallback;
}

// The 35 bytes of a structured frame that do not depend on the ciphertext (zstd_pack40 layout, codec.cpp): frame header,
// block A header + raw-literals header + its one sequence, word-block header + raw-literals header, sequence count + tables.
// One routine writes them (k_ct_pack40) or compares them (k_unpack40): a frame whose fixed bytes differ is not a structured
// frame -- any zstd decoder would read something else or reject it -- and goes back to the host path.
template <bool kWrite>
__device__ __forceinline__ bool frame40_fixed(uint8_t *f) {
    bool ok = true;
    const auto put = [&](size_t at, uint8_t v) {
        if (kWrite) f[at] = v;
        else ok = ok && f[at] == v;
    };
    const uint8_t h[9] = {0x28, 0xB5, 0x2F, 0xFD, 0xA0, (uint8_t)kCtPayloadBytes, (uint8_t)(kCtPayloadBytes >> 8),
                          (uint8_t)(kCtPayloadBytes >> 16), (uint8_t)(kCtPayloadBytes >> 24)};  // magic, single segment, content size
    for (int k = 0; k < 9; k++) put(k, h[k]);
    const uint32_t bh = (2u << 1) | ((2 + 110 + 7) << 3);  // block A: compressed block of 2 + 110 + 7 bytes
    put(9, (uint8_t)bh), put(10, (uint8_t)(bh >> 8)), put(11, (uint8_t)(bh >> 16));
    const uint32_t lh = (1u << 2) | (110u << 4);  // 110 raw literals
    put(12, (uint8_t)lh), put(13, (uint8_t)(lh >> 8));
    const uint32_t bits = (110 - 64) | (3u << 6) | (1u << 9);
    const uint8_t sq[7] = {0x01, 0x54, 25, 3, 0, (uint8_t)bits, (uint8_t)(bits >> 8)};  // one sequence: LL 110, ML 3, offset 8
    for (int k = 0; k < 7; k++) put(14 + 110 + k, sq[k]);
    constexpr uint32_t m = (uint32_t)kCodecCtWords - 2, body = 3 + 5 * m + 2 + 5;  // word block: 16382 words, last block
    const uint32_t bh2 = 1u | (2u << 1) | (body << 3);
    const size_t g = 9 + 122;
    put(g, (uint8_t)bh2), put(g + 1, (uint8_t)(bh2 >> 8)), put(g + 2, (uint8_t)(bh2 >> 16));
    const uint32_t lh2 = (3u << 2) | ((5 * m) << 4);
    put(g + 3, (uint8_t)lh2), put(g + 4, (uint8_t)(lh2 >> 8)), put(g + 5, (uint8_t)(lh2 >> 16));
    const size_t t = g + 6 + 5 * (size_t)m;
    put(t, (uint8_t)((m >> 8) + 0x80)), put(t + 1, (uint8_t)m);
    const uint8_t tail[5] = {0x54, 5, 0, 0, 0x01};  // RLE tables, (LL 5, ML 3, repeat offset 1), end marker
    for (int k = 0; k < 5; k++) put(t + 2 + k, tail[k]);
    return ok;
}

// structured frames: literals are at two fixed places of the frame; block (j, 0) also verifies the frame's length and every
// fixed byte, the other blocks the residues
__global__ void __launch_bounds__(256) k_unpack40(const uint8_t *frames, const CodecJob *jobs, int32_t *status, const uint8_t *prefix,
                                                  u64 *dst_a, u64 *dst_b) {
    const int j = blockIdx.x;
    const CodecJob job = jobs[j];
    if (job.kind != kJobPacked) return;
    const uint8_t *f = frames + job.src_off;
    __shared__ int bad;
    if (threadIdx.x == 0) bad = 0;
    __syncthreads();
    int mybad = 0;
    const uint8_t *la = f + 9 + 3 + 2;  // block A literals: prefix, word 0 (8 bytes), low 5 bytes of word 1
    if (blockIdx.y == 0 && threadIdx.x < kCtPrefixBytes && threadIdx.x != 77 && la[threadIdx.x] != prefix[threadIdx.x]) mybad = 1;
    if (blockIdx.y == 0 && threadIdx.x == 128 && (job.src_len != kPackedFrameBytes || !frame40_fixed<false>(const_cast<uint8_t *>(f))))
        mybad = 1;
    u64 *dst = (job.operand ? dst_b : dst_a) + (size_t)job.slot * kCodecCtWords;
    const uint8_t *lw = f + 9 + (3 + 2 + 110 + 7) + 3 + 3;  // literals of words 2..
    const int lo = blockIdx.y * kWordsPerBlock;
    for (int i = lo + threadIdx.x; i < lo + kWordsPerBlock; i += 256) {
        u64 w = 0;
        if (i >= 2) {
            const uint8_t *s = lw + 5 * (size_t)(i - 2);
            w = (u64)s[0] | (u64)s[1] << 8 | (u64)s[2] << 16 | (u64)s[3] << 24 | (u64)s[4] << 32;
        } else {
            const uint8_t *s = la + kCtPrefixBytes + 8 * i;
            const int nb = i == 0 ? 8 : 5;
            for (int k = 0; k < nb; k++) w |= (u64)s[k] << (8 * k);
        }
        if (w >= (((i >> 12) & 1) ? kQ1 : kQ0)) mybad = 1;
        dst[i] = w;
    }
    if (mybad) atomicOr(&bad, 1);
    __syncthreads();
    if (threadIdx.x == 0 && bad) status[j] = kJobFallback;
}

// words -> complete structured frame (kPackedFrameBytes); flag = 1 when the first 16 words are equal (the host writer hands
// constant data to libzstd, and so must the caller).  Output j starts at out + j * out_stride with the `head_len` bytes of
// `head` (the bincode + SEAL envelope of a complete Ciphertext, or nothing), and its frame follows them.
__global__ void __launch_bounds__(256) k_ct_pack40(const u64 *words, uint8_t *out, size_t out_stride, const uint8_t *head, int head_len,
                                                   int32_t *constant_flag, const uint8_t *prefix) {
    const int j = blockIdx.x;
    const u64 *w = words + (size_t)j * kCodecCtWords;
    uint8_t *f = out + (size_t)j * out_stride + head_len;
    if (blockIdx.y == 0 && (int)threadIdx.x < head_len) f[(int)threadIdx.x - head_len] = head[threadIdx.x];  // head_len <= 256
    if (blockIdx.y == 0 && threadIdx.x == 0) {
        frame40_fixed<true>(f);
        u64 diff = 0;
        for (int k = 1; k < 16; k++) diff |= w[k] ^ w[0];
        constant_flag[j] = diff == 0;
    }
    uint8_t *la = f + 14;
    if (blockIdx.y == 0 && threadIdx.x < kCtPrefixBytes) la[threadIdx.x] = prefix[threadIdx.x];
    uint8_t *lw = f + 9 + 122 + 6;
    const int lo = blockIdx.y * kWordsPerBlock;
    for (int i = lo + threadIdx.x; i < lo + kWordsPerBlock; i += 256) {
        const u64 v = w[i];
        if (i >= 2) {
            uint8_t *d = lw + 5 * (size_t)(i - 2);
            d[0] = (uint8_t)v, d[1] = (uint8_t)(v >> 8), d[2] = (uint8_t)(v >> 16), d[3] = (uint8_t)(v >> 24), d[4] = (uint8_t)(v >> 32);
        } else {
            uint8_t *d = la + kCtPrefixBytes + 8 * i;
            const int nb = i == 0 ? 8 : 5;
            for (int k = 0; k < nb; k++) d[k] = (uint8_t)(v >> (8 * k));
        }
    }
}
}  // namespace

size_t codec_work_bytes() { return sizeof(JobScratch); }

cudaError_t launch_codec_inflate(const uint8_t *frames, uint8_t *payloads, const CodecJob *jobs, int32_t *status, void *work,
                                 const uint8_t *prefix, u64 *dst_a, u64 *dst_b, int n_jobs, bool any_zstd, bool any_packed,
                                 bool any_payload, cudaStream_t s) {
    if (n_jobs == 0) return cudaSuccess;
    cudaError_t ce = cudaMemsetAsync(status, 0, (size_t)n_jobs * sizeof(int32_t), s);  // kJobPending
    if (ce != cudaSuccess) return ce;
    if (any_zstd) {
        static std::atomic<int> configured{0};  // (per process; the attributes are per function and device-independent in effect)
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (!((configured.load() >> dev) & 1)) {
            cudaError_t e = cudaFuncSetAttribute(k_zd3_exec, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)zd3::kExecSmem);
            if (e != cudaSuccess) return e;
            configured.fetch_or(1 << dev);
        }
        k_zd2_parse<<<(n_jobs + 31) / 32, 32, 0, s>>>(frames, jobs, (JobScratch *)work, n_jobs);
        k_zd3_huf<<<(n_jobs + 31) / 32, 128, 0, s>>>(frames, jobs, (JobScratch *)work, n_jobs);
        k_zd3_seq<<<(n_jobs + zd3::kSeqFrames - 1) / zd3::kSeqFrames, 32, zd3::kSeqSmem, s>>>(frames, jobs, (JobScratch *)work, n_jobs);
        k_zd3_exec<<<n_jobs < 2 * sms ? n_jobs : 2 * sms, zd3::kExecThreads, zd3::kExecSmem, s>>>(frames, payloads, jobs, status,
                                                                                                    (JobScratch *)work, n_jobs);
        g_codec_launches.fetch_add(4, std::memory_order_relaxed);
    }
    if ((any_zstd || any_payload) && dst_a) {  // (the standalone inflate entry point stops at the payloads)
        k_ct_unpack<<<dim3(n_jobs, kSplit), 256, 0, s>>>(payloads, jobs, status, prefix, dst_a, dst_b);
        g_codec_launches.fetch_add(1, std::memory_order_relaxed);
    }
    if (any_packed) {
        k_unpack40<<<dim3(n_jobs, kSplit), 256, 0, s>>>(frames, jobs, status, prefix, dst_a, dst_b);
        g_codec_launches.fetch_add(1, std::memory_order_relaxed);
    }
    return cudaGetLastError();
}

cudaError_t launch_codec_pack(const u64 *words, uint8_t *frames, int32_t *constant_flag, const uint8_t *prefix, int n, cudaStream_t s) {
    return launch_codec_pack(words, frames, kPackedFrameStride, nullptr, 0, constant_flag, prefix, n, s);
}

cudaError_t launch_codec_pack(const u64 *words, uint8_t *out, size_t out_stride, const uint8_t *head, int head_len, int32_t *constant_flag,
                              const uint8_t *prefix, int n, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    if (head_len < 0 || head_len > kPackHeadMax || out_stride < (size_t)head_len + kPackedFrameBytes) return cudaErrorInvalidValue;
    k_ct_pack40<<<dim3(n, kSplit), 256, 0, s>>>(words, out, out_stride, head, head_len, constant_flag, prefix);
    g_codec_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError();
}

uint64_t codec_launch_count() { return g_codec_launches.load(); }

}  // namespace fheb
