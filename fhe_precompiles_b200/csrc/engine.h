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

// the keys of a key switch with a key per op: op i of a chunk runs under key key_index[i] of n_keys
struct RelinKeys {
    const uint64_t *const *raw = nullptr;  // device array of n_keys device pointers to SEAL-form keys [2][2][3][N] (split tails)
    size_t n_keys = 0;
    uint64_t *prepared = nullptr;  // [n_keys][12][N] dual-base keys (fused tails), filled by the first chunk that runs them
    bool ready = false;            // `prepared` holds the keys
    const int32_t *key_index = nullptr;  // device ints of the chunk's ops (not checked)
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
    // a tile's ct-ct multiplies under more than one key: its distinct keys and each slot's index into them (cap entries each)
    const uint64_t **h_rk_ptrs = nullptr, **d_rk_ptrs = nullptr;
    int32_t *h_rk_index = nullptr, *d_rk_index = nullptr;
    bool busy = false;
    // device codec staging for tiles (allocated when a tile first uses it): compressed operand frames in, structured frames out
    size_t codec_cap = 0;
    uint8_t *h_frames = nullptr, *d_frames = nullptr, *h_payloads = nullptr, *d_payloads = nullptr, *h_outframes = nullptr, *d_outframes = nullptr;
    const uint8_t *d_prefix = nullptr;  // the engine's canonical ciphertext prefix on this lane's device
    struct CodecJob *h_jobs = nullptr, *d_jobs = nullptr;
    int32_t *h_status = nullptr, *d_status = nullptr;  // [2 * cap] job status, then [cap] constant-result flags
    void *d_work = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};  // call-breakdown timing (created on first use)
    // CUDA graphs of the single-call fast path (copies + codec kernels + arithmetic), captured once per call shape and relin
    // key on this lane's buffers; dropped whenever the buffers are reallocated
    struct CallGraph {
        int op, shape, route0, route1;
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

// one call of the threshold-network precompiles (encrypt_*, reencrypt_*, decrypt_*) inside a tile of the batch surface
enum class Threshold : int { Encrypt = 0, Reencrypt = 1, Decrypt = 2 };
struct ThresholdItem {
    Threshold op;
    Kind kind;
    Span in;
    std::vector<uint8_t> out;
    int32_t rc = 0;
    bool take_malloc = false;  // as TileItem
    uint8_t *out_malloc = nullptr;
    size_t out_malloc_len = 0;
    bool single = false;  // set by threshold_tile: the tile did not take the call, whose caller runs it as the single call
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
    // the calling thread is one of many tile workers: binary_tile keeps its per-call loops on it instead of sharing them with the pool
    static void set_thread_serial_loops(bool on);
    // ... or may share them with at most `threads` - 1 pool threads (0: no limit): a batch divides its thread budget among its workers
    static void set_thread_loop_width(size_t threads);
    static constexpr size_t kZstdTileMinBatch = 2048;
    // Big tiles: a batch of >= kZstdTileMinBatch calls runs as a few tiles of an eighth of itself, between 256 and 1,024 calls
    // (0: smaller batches), each staging its calls on the whole host pool and launching thousands of operand frames at once (the
    // device zstd decoder's rate grows with the frames per launch: 183 k frames/s at 1,024, 431 k at 8,192).  Never more than
    // n / 2: a batch in big tiles has at least two of them.
    static size_t big_tile_ops_for(size_t n) {
        if (n < kZstdTileMinBatch) return 0;
        size_t b = 256;
        while (b < 1024 && 2 * b <= n / 8) b *= 2;
        return b;
    }
    // per-call phase timing of binary_tile (host clock around the codec phases, CUDA events around the copies and the
    // kernels on the lane's stream); off by default
    void set_call_timing(bool on) { call_timing_ = on; }
    static const CallBreakdown &last_call_breakdown();

    // device-resident batched entry points (pointers are device memory on `device`)
    void mul_relin(int device, const uint64_t *a, const uint64_t *b, const uint64_t *rk, uint64_t *out, size_t n,
                   cudaStream_t s);
    void multiply(int device, const uint64_t *a, const uint64_t *b, uint64_t *out3, size_t n, cudaStream_t s);
    void relinearize(int device, const uint64_t *c3, const uint64_t *rk, uint64_t *out, size_t n, cudaStream_t s);
    // the same with a key per row: rks [n_keys][2][2][3][N], key_index [n] device ints in [0, n_keys) (not checked); row i is
    // bit for bit mul_relin / relinearize of that row under rks[key_index[i]].  All n_keys keys are prepared, once per call, into
    // n_keys x 12 limbs of the stream's scratch arena (which keeps its size): the caller passes the keys its rows use.
    void mul_relin_keyed(int device, const uint64_t *a, const uint64_t *b, const uint64_t *rks, size_t n_keys, const int32_t *key_index,
                         uint64_t *out, size_t n, cudaStream_t s);
    void relinearize_keyed(int device, const uint64_t *c3, const uint64_t *rks, size_t n_keys, const int32_t *key_index, uint64_t *out,
                           size_t n, cudaStream_t s);

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
    // The same from / to complete sunscreen Ciphertexts of `kind`, in whatever form the precompiles accept (libzstd, structured,
    // zlib or uncompressed SEAL blobs) and write.  upload: status[i] = 0 or the code c_fhe_add_cipherK_cipherK returns for
    // ciphertext i as its first operand (the words of that row are then undefined).  download: outputs[i] malloc'ed, byte for byte
    // what a precompile of `kind` returns for these words under the current zstd writer; status[i] = -1 where a row failed
    // (its message in *row_error).  Synchronous, in chunks of kXferChunk over the two transfer slots.
    void upload_ciphertexts(int device, Kind kind, const uint8_t *const *cts, const size_t *lens, size_t n, uint64_t *d_words,
                            int32_t *status);
    void download_ciphertexts(int device, Kind kind, const uint64_t *d_words, size_t n, uint8_t **outputs, int64_t *output_lengths,
                              int32_t *status, std::string *row_error);

    // Optional per-kernel timing of mul_relin(): CUDA events around every launch on the caller's stream.
    // kernel ids: see kKernelNames.  report() synchronises the device.
    static constexpr int kNumTimedKernels = 16;
    void set_kernel_timing(bool on);
    void kernel_timing_report(int device, double ms[kNumTimedKernels], uint64_t launches[kNumTimedKernels]);

    // threshold-network simulation API (fhe.rs:594-779) against the embedded network keys
    int32_t encrypt(Kind kind, Span in, Span net_pub, Span net_pri, std::vector<uint8_t> *out);
    int32_t reencrypt(Kind kind, Span in, Span net_pub, Span net_pri, std::vector<uint8_t> *out);
    int32_t decrypt(Kind kind, Span in, Span net_pub, Span net_pri, std::vector<uint8_t> *out);
    // `cnt` independent threshold calls on ONE lane: one batched decryption over every decrypt_* / reencrypt_* operand and one
    // batched encryption (a key per row) over every encrypt_* / reencrypt_* result.  Per-call results and error codes are exactly
    // those of the three functions above.  A call whose operand is not perfectly ordinary (or a tile of one) is left marked
    // `single`, with no result: the caller runs it as the single call after this returns.
    void threshold_tile(ThresholdItem *items, size_t cnt, Span net_pub, Span net_pri);

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
    // the same with a key per op: pks [k][2][3][N], key_index [n] ints in [0, k) (device data, not checked)
    void encrypt_keyed_device(int device, const uint64_t *pks, const int32_t *key_index, const uint16_t *plain, const uint64_t *seeds,
                              uint64_t *ct, size_t n, cudaStream_t s);
    // exhausted (optional, [n] ints on the device): 1 where the invariant noise budget is 0 (the plaintext is then garbage)
    void decrypt_device(int device, const uint64_t *ct, const uint64_t *sk, uint16_t *plain, size_t n, cudaStream_t s,
                        int32_t *exhausted = nullptr);

   private:
    Engine();
    void create_lanes();
    void ensure_capacity(Lane *lane, size_t cap);
    void ensure_codec(Lane *lane);
    bool single_call_fast(Lane *lane, TileItem &it, bool timed, std::chrono::steady_clock::time_point t_start);
    // threshold_tile's device passes on `lane`
    void threshold_on_lane(Lane *lane, ThresholdItem *items, size_t cnt, Span net_pub, Span net_pri);
    void drop_graphs(Lane *lane);
    size_t tile_ops_ = 16;
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
        size_t chunk = 0;
        uint64_t *d_rk = nullptr;
        int32_t *h_status = nullptr;  // pinned, 3 per op of the largest call so far
        size_t h_status_cap = 0;
        PipeSlot slot[kPipeSlots];
        std::mutex mu;
    };
    std::vector<std::unique_ptr<HostPipe>> pipes_;
    // the device's host pipeline with its streams and per-slot chunk buffers, `rk` uploaded; returns with `lk` holding its mu
    HostPipe &host_pipe(int device, const uint64_t *rk, std::unique_lock<std::mutex> &lk);
    // the 97 bytes every valid ciphertext payload starts with (canonical_ct_prefix), on `device`: the codec kernels check them
    std::vector<uint8_t *> d_prefix_;
    std::mutex prefix_mu_;
    const uint8_t *ct_prefix(int device);
    // staging of upload_frames / download_frames: two slots per device, alternating chunks
    struct XferSlot {
        cudaStream_t stream = nullptr;
        uint8_t *d_frames = nullptr;  // chunk * stride + 2 pads (upload) or chunk * kPackedFrameStride (download)
        size_t d_frames_bytes = 0;
        struct CodecJob *d_jobs = nullptr, *h_jobs = nullptr;
        int32_t *d_status = nullptr;
        // upload_ciphertexts / download_ciphertexts: pinned mirror of d_frames (the scattered ciphertexts are gathered here, then
        // cross PCIe in one copy), and the device zstd decoder's workspace; both allocated on first use
        uint8_t *h_stage = nullptr;
        size_t h_stage_bytes = 0;
        void *d_work = nullptr;
    };
    struct XferPipe {
        uint8_t *d_head = nullptr;  // download_ciphertexts: the envelope in front of every structured frame (kPackHeadMax bytes)
        int32_t *h_status = nullptr;
        size_t h_status_cap = 0;
        XferSlot slot[2];
        std::mutex mu;
    };
    static constexpr size_t kXferChunk = 256;
    std::vector<std::unique_ptr<XferPipe>> xfers_;
    XferPipe &xfer_pipe(int device, size_t n, size_t slot_bytes);
    void xfer_host_stage(XferPipe &X, size_t bytes);  // XferSlot::h_stage of at least `bytes`; X.mu held

    struct TimedLaunch {
        int kernel;
        cudaEvent_t e0, e1;
    };
    bool timing_ = false;
    void enqueue_mul(const uint64_t *a, const uint64_t *b, const ScratchMap &m, size_t c, cudaStream_t s, bool timed);
    // keys (optional): a key per op instead of rk
    void enqueue_relin(const uint64_t *c3, const uint64_t *rk, uint64_t *out, const ScratchMap &m, size_t c, cudaStream_t s,
                       bool timed, RelinKeys *keys = nullptr);
    // mul_relin_keyed (a, b) or relinearize_keyed (c3)
    void keyed_chunks(int device, const uint64_t *a, const uint64_t *b, const uint64_t *c3, const uint64_t *rks, size_t n_keys,
                      const int32_t *key_index, uint64_t *out, size_t n, cudaStream_t s);
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
