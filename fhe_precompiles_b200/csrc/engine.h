// Dispatcher between the byte surface and the kernels: what FheApp (fhe.rs:56-780) + sunscreen's
// Runtime::run do in the reference.  One process-wide Engine, re-entrant like the reference's
// `FHE: Lazy<FheApp>` (testnet.rs:25).  There is no CPU path: every op runs on a CUDA device or fails.
#pragma once
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdint>
#include <memory>
#include <mutex>
#include <vector>

#include "codec.h"
#include "context.h"

namespace fheb {

enum class Op : int { Add = 0, Sub = 1, Mul = 2 };
enum class Shape : int { CtCt = 0, CtPt = 1, PtCt = 2 };

// limbs of per-op scratch for multiply+relinearise:
// tensor (15) + size-3 result (6) + key-switch (6) + NTT-domain operands (20) + NTT-domain digits (6)
constexpr size_t kScratchLimbsPerOp = 15 + 6 + 6 + 20 + 6;

// offsets (in limbs, per chunk of `c` ops) of the scratch regions
struct ScratchMap {
    uint64_t *tens, *c3, *ks, *nttbuf, *dig;
    ScratchMap(uint64_t *base, size_t c)
        : tens(base), c3(tens + c * 15 * kN), ks(c3 + c * 6 * kN), nttbuf(ks + c * 6 * kN), dig(nttbuf + c * 20 * kN) {}
};

// A lane = one stream + staging for `cap` calls (1 until a tile of the batch surface needs more).
struct Lane {
    int device = 0;
    cudaStream_t stream = nullptr;
    size_t cap = 0;
    uint64_t *h_a = nullptr, *h_b = nullptr, *h_out = nullptr;  // pinned, cap * kCtWords each
    uint16_t *h_plain = nullptr;                                // pinned, cap * kN
    uint64_t *d_a = nullptr, *d_b = nullptr, *d_out = nullptr, *d_scratch = nullptr;
    uint16_t *d_plain = nullptr;
    bool busy = false;
    // device codec staging for tiles (allocated when a tile first uses it): compressed operand frames in, structured frames out
    size_t codec_cap = 0;
    uint8_t *h_frames = nullptr, *d_frames = nullptr, *h_payloads = nullptr, *d_payloads = nullptr, *h_outframes = nullptr, *d_outframes = nullptr;
    uint8_t *d_prefix = nullptr;
    struct CodecJob *h_jobs = nullptr, *d_jobs = nullptr;
    int32_t *h_status = nullptr, *d_status = nullptr;  // [2 * cap] job status, then [cap] constant-result flags
    void *d_work = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};  // call-breakdown timing (created on first use)
    // CUDA graphs of the single-call fast path (copies + codec kernels + arithmetic), captured once per call shape and relin
    // key on this lane's buffers; dropped whenever the buffers are reallocated
    struct CallGraph {
        int op, shape, kind0, kind1;
        const uint64_t *rk;
        cudaGraphExec_t exec;
        uint64_t launches;  // kernels inside, for the launch counter
    };
    std::vector<CallGraph> graphs;
};

// where the time of the last binary call (or tile) on this thread went, microseconds
struct CallBreakdown {
    double unpack_key_us = 0, decode_us = 0, h2d_us = 0, kernels_us = 0, d2h_us = 0, encode_us = 0, total_us = 0;
};

// one call of the 36 binary precompiles inside a tile of the batch surface
struct TileItem {
    Op op;
    Shape shape;
    Kind kind;
    Span in;
    std::vector<uint8_t> out;
    int32_t rc = 0;
    // a result the tile already wrote into a malloc'ed buffer (batch workers: handed to the caller as it is, no second copy);
    // used only when `take_malloc` was set by the caller of binary_tile, who then owns the buffer
    bool take_malloc = false;
    uint8_t *out_malloc = nullptr;
    size_t out_malloc_len = 0;
};

struct KeyEntry {
    std::vector<uint8_t> bytes;  // exact PublicKey bytes this entry was parsed from
    uint64_t tag = 0;            // cheap pre-filter
    bool has_relin = false;
    std::vector<uint64_t> rk;    // host copy [2][2][3][N]
    std::vector<uint64_t> pk;    // host copy [2][3][N]
    std::vector<uint64_t *> d_rk;  // per device, lazily uploaded
    std::vector<uint64_t *> d_pk;
    uint64_t last_use = 0;
    int users = 0;  // calls currently holding device pointers of this entry (guarded by Engine::key_mu_); pinned against eviction
};

class Engine;
// RAII pin on a cached key: the entry's device buffers stay allocated until every holder is gone
class KeyPin {
   public:
    KeyPin() = default;
    KeyPin(Engine *e, KeyEntry *k) : e_(e), k_(k) {}
    KeyPin(const KeyPin &) = delete;
    KeyPin &operator=(const KeyPin &) = delete;
    KeyPin(KeyPin &&o) noexcept : e_(o.e_), k_(o.k_) { o.k_ = nullptr; }
    KeyPin &operator=(KeyPin &&o) noexcept;
    ~KeyPin() { release(); }
    void release();

   private:
    Engine *e_ = nullptr;
    KeyEntry *k_ = nullptr;
};

class Engine {
   public:
    static Engine &get();

    // the 36 binary precompiles: bytes in -> bytes out (lib.rs error code)
    int32_t binary_op(Op op, Shape shape, Kind kind, Span in, std::vector<uint8_t> *out);
    // `cnt` independent binary precompile calls on ONE lane: operands decoded into adjacent staging slots, one H2D / D2H
    // per operand array and one batched kernel sequence per (operation, relin key) class instead of per call.
    // Per-call results and error codes are exactly those of binary_op (which is a tile of one).
    void binary_tile(TileItem *items, size_t cnt);
    size_t tile_ops() const { return tile_ops_; }
    size_t lane_device_count() const { return lane_devices_.size(); }  // GPUs the byte surface spreads its lanes over
    // tile size for a batch of n calls: large batches run in tiles big enough for the device zstd decoder to take their operand
    // frames (device_zstd_ == 2), everything else in tile_ops_
    size_t tile_ops_for(size_t n) const {
        return (device_codec_ && device_zstd_ == 2 && n >= zstd_tile_min_batch_ && zstd_tile_ops_ > tile_ops_) ? zstd_tile_ops_ : tile_ops_;
    }
    // the calling thread is one of many tile workers: binary_tile keeps its per-call loops on it instead of sharing them with the pool
    static void set_thread_serial_loops(bool on);
    // ... or may share them with at most `threads` - 1 pool threads (0: no limit): a batch divides its thread budget among its workers
    static void set_thread_loop_width(size_t threads);
    // tile size of a large batch: big tiles put thousands of operand frames in flight per launch (the device zstd decoder's
    // throughput comes from frames in flight) and their staging loops are shared with the host pool
    // Big tiles: a large batch runs as a few tiles of this many calls, each staging its calls on the whole host pool and
    // launching thousands of operand frames at once (the device zstd decoder's rate grows with the frames per launch: 183 k
    // frames/s at 1,024, 431 k at 8,192).  FHE_B200_BIG_TILE_OPS fixes the size (0 there: never); by default a batch of
    // >= 2,048 calls takes an eighth of itself, between 256 and 1,024 calls.
    size_t big_tile_ops_for(size_t n) const {
        if (big_tile_set_) return big_tile_ops_;
        if (!(device_codec_ && device_zstd_ == 2 && n >= zstd_tile_min_batch_)) return 0;
        size_t b = 256;
        while (b < 1024 && 2 * b <= n / 8) b *= 2;
        return b;
    }
    bool device_codec() const { return device_codec_; }
    // per-call phase timing of binary_tile (host clock around the codec phases, CUDA events around the copies and the
    // kernels on the lane's stream); off by default
    void set_call_timing(bool on) { call_timing_ = on; }
    static const CallBreakdown &last_call_breakdown();

    // device-resident batched entry points (pointers are device memory on `device`)
    void mul_relin(int device, const uint64_t *a, const uint64_t *b, const uint64_t *rk, uint64_t *out, size_t n,
                   cudaStream_t s);
    void multiply(int device, const uint64_t *a, const uint64_t *b, uint64_t *out3, size_t n, cudaStream_t s);
    void relinearize(int device, const uint64_t *c3, const uint64_t *rk, uint64_t *out, size_t n, cudaStream_t s);

    // host-buffer batched entry point: a, b, out are host memory (pinned for full PCIe rate), rk host words.
    // H2D, kernels and D2H of consecutive chunks overlap on `kPipeSlots` streams.  Synchronous.
    void mul_relin_host(int device, const uint64_t *a, const uint64_t *b, const uint64_t *rk, uint64_t *out, size_t n);
    // the same on serialized operands: structured zstd frames (what this library writes) in, structured frames out
    void mul_relin_frames(int device, const uint8_t *fa, const uint8_t *fb, size_t stride, const uint64_t *rk, uint8_t *fout, size_t n,
                          int32_t *status);

    // Device-resident ciphertexts from / to serialized form (structured frames), so that a chain of device-resident ops pays
    // PCIe once at each end: frames (host) -> validated limb arrays on the device, and back.  Synchronous, chunk-pipelined.
    void upload_frames(int device, const uint8_t *frames, size_t stride, size_t n, uint64_t *d_words, int32_t *status);
    void download_frames(int device, const uint64_t *d_words, size_t n, uint8_t *out_frames, int32_t *status);

    // Optional per-kernel timing of mul_relin(): CUDA events around every launch on the caller's stream.
    // kernel ids: see kKernelNames.  report() synchronises the device.
    static constexpr int kNumTimedKernels = 16;
    void set_kernel_timing(bool on);
    void kernel_timing_report(int device, double ms[kNumTimedKernels], uint64_t launches[kNumTimedKernels]);

    // threshold-network simulation API (fhe.rs:594-779) against the embedded network keys
    int32_t encrypt(Kind kind, Span in, Span net_pub, Span net_pri, std::vector<uint8_t> *out);
    int32_t reencrypt(Kind kind, Span in, Span net_pub, Span net_pri, std::vector<uint8_t> *out);
    int32_t decrypt(Kind kind, Span in, Span net_pub, Span net_pri, std::vector<uint8_t> *out);

    // scratch arena for `ops` concurrent multiply+relin ops, one per (device, caller stream): grown on demand, leased while
    // a caller enqueues, evicted (after synchronising its stream) when more than FHE_B200_SCRATCH_ARENAS are idle on a device
    struct StreamState {
        int device = 0;
        cudaStream_t stream = nullptr;
        uint64_t *p = nullptr;
        size_t ops = 0;
        int users = 0;
        uint64_t last_use = 0;
    };
    StreamState *lease_scratch(int device, cudaStream_t s, size_t ops);
    void release_scratch(StreamState *st);
    size_t chunk_ops() const { return chunk_ops_; }
    size_t set_chunk_ops(long long ops);  // ops <= 0 only queries; returns the previous value
    int n_devices() const { return n_devices_; }

    // relin key for the PublicKey bytes, parsed + validated once and cached by content
    // `pin` keeps the entry (and its device buffers) alive until it is destroyed
    int32_t relin_key(Span pk, int device, const uint64_t **d_rk, bool need_relin, KeyPin *pin);
    // encryption key [2][3][N] on `device` for the PublicKey bytes (same cache)
    int32_t public_key(Span pk, int device, const uint64_t **d_pk, KeyPin *pin);
    void unpin_key(KeyEntry *k);
    // device-resident batched encrypt / decrypt (pointers on `device`)
    void encrypt_device(int device, const uint64_t *pk, const uint16_t *plain, const uint64_t *seeds, uint64_t *ct, size_t n,
                        cudaStream_t s);
    // exhausted (optional, [n] ints on the device): 1 where the invariant noise budget is 0 (the plaintext is then garbage)
    void decrypt_device(int device, const uint64_t *ct, const uint64_t *sk, uint16_t *plain, size_t n, cudaStream_t s,
                        int32_t *exhausted = nullptr);

   private:
    Engine();
    void create_lanes();
    void ensure_capacity(Lane *lane, size_t cap);
    void ensure_codec(Lane *lane);
    bool single_call_fast(Lane *lane, TileItem &it, bool timed, std::chrono::steady_clock::time_point t_start);
    bool device_codec_ = true;  // FHE_B200_DEVICE_CODEC=0: tiles decode and encode everything on the host
    bool call_graphs_ = true;   // FHE_B200_CALL_GRAPHS=0: the single-call fast path launches its kernels one by one
    void drop_graphs(Lane *lane);
    // libzstd-written operand frames inflated on the GPU (codec_kernels.cu): 0 never, 1 always, 2 (default) when a tile brings at
    // least device_zstd_min_frames_ of them; host_inflate_pct_ % of those frames are inflated by the host cores meanwhile
    int device_zstd_ = 2;
    size_t device_zstd_min_frames_ = 128, host_inflate_pct_ = 0;
    size_t zstd_tile_ops_ = 128, zstd_tile_min_batch_ = 2048;
    size_t tile_ops_ = 16, big_tile_ops_ = 0;
    bool big_tile_set_ = false;
    bool helper_decode_ = true;  // FHE_B200_HELPER_DECODE=0 turns the helper-thread inflate of single calls off
    std::atomic<bool> call_timing_{false};
    std::vector<int> lane_devices_;
    Lane *acquire_lane();
    void release_lane(Lane *);

    int n_devices_ = 0;
    size_t chunk_ops_ = 4096;
    std::vector<std::unique_ptr<Lane>> lanes_;
    std::mutex lane_mu_;
    std::condition_variable lane_cv_;

    KeyEntry *find_or_parse_key(Span pk, int32_t *rc);  // returns the entry PINNED (users + 1); takes key_mu_ itself
    const uint64_t *network_sk(int device, Span net_pri);
    int32_t encrypt_plain(Kind kind, Span scalar, Span pk_bytes, const uint64_t seed[8], CipherView *view, Lane *lane,
                          std::vector<uint8_t> *out);
    std::vector<uint64_t *> d_net_sk_;
    std::mutex sk_mu_;
    std::mutex key_mu_;
    std::vector<std::unique_ptr<KeyEntry>> keys_;
    uint64_t key_clock_ = 0;

    static constexpr int kPipeSlots = 3;
    struct PipeSlot {
        cudaStream_t stream = nullptr;
        uint64_t *d_a = nullptr, *d_b = nullptr, *d_out = nullptr, *d_scratch = nullptr;
        // mul_relin_frames: staged operand frames, result frames, codec jobs / status
        uint8_t *d_frames = nullptr, *d_outframes = nullptr;
        struct CodecJob *d_jobs = nullptr;
        int32_t *d_status = nullptr;
        size_t frame_stride = 0;
    };
    struct HostPipe {
        bool ready = false;
        size_t chunk = 0;
        uint64_t *d_rk = nullptr;
        uint8_t *d_prefix = nullptr;
        int32_t *h_status = nullptr;  // pinned, 3 per op of the largest call so far
        size_t h_status_cap = 0;
        PipeSlot slot[kPipeSlots];
        std::mutex mu;
    };
    std::vector<std::unique_ptr<HostPipe>> pipes_;
    // staging of upload_frames / download_frames: two slots per device, alternating chunks
    struct XferSlot {
        cudaStream_t stream = nullptr;
        uint8_t *d_frames = nullptr;  // chunk * stride + 2 pads (upload) or chunk * kPackedFrameStride (download)
        size_t d_frames_bytes = 0;
        struct CodecJob *d_jobs = nullptr, *h_jobs = nullptr;
        int32_t *d_status = nullptr;
    };
    struct XferPipe {
        uint8_t *d_prefix = nullptr;
        int32_t *h_status = nullptr;
        size_t h_status_cap = 0;
        XferSlot slot[2];
        std::mutex mu;
    };
    static constexpr size_t kXferChunk = 256;
    std::vector<std::unique_ptr<XferPipe>> xfers_;
    XferPipe &xfer_pipe(int device, size_t n, size_t slot_bytes);

    struct TimedLaunch {
        int kernel;
        cudaEvent_t e0, e1;
    };
    bool timing_ = false;
    void enqueue_mul(const uint64_t *a, const uint64_t *b, const ScratchMap &m, size_t c, cudaStream_t s, bool timed);
    void enqueue_relin(const uint64_t *c3, const uint64_t *rk, uint64_t *out, const ScratchMap &m, size_t c, cudaStream_t s,
                       bool timed);
    void timed_launch(int kernel, cudaStream_t s, bool timed, cudaError_t e0, const char *what);
    std::vector<TimedLaunch> timed_;
    std::mutex timed_mu_;
    std::vector<cudaEvent_t> event_pool_;
    cudaEvent_t take_event();

    void free_stream_state(StreamState &v);
    std::vector<std::unique_ptr<StreamState>> stream_states_;
    uint64_t arena_clock_ = 0;
    std::condition_variable arena_cv_;
    std::mutex arena_mu_;
};

void cuda_throw(cudaError_t e, const char *what);
uint64_t launch_count();

}  // namespace fheb
