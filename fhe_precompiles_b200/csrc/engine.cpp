// See engine.h.
#include "engine.h"

#include <algorithm>
#include <chrono>
#include <functional>

#include "codec_stage.h"
#include "host_pool.h"

#include <cstdlib>
#include <cstring>
#include <map>
#include <stdexcept>
#include <string>
#include <thread>

#include "kernels.h"

namespace fheb {

void cuda_throw(cudaError_t e, const char *what) {
    if (e != cudaSuccess)
        throw std::runtime_error(std::string("fhe_b200: CUDA error in ") + what + ": " + cudaGetErrorString(e));
}

namespace {
size_t env_size(const char *name, size_t dflt) {
    const char *v = getenv(name);
    if (!v || !*v) return dflt;
    long long x = atoll(v);
    return x > 0 ? (size_t)x : dflt;
}
uint64_t cheap_tag(Span s) {
    // length + 4 sampled words: a pre-filter only, equality is decided by memcmp
    uint64_t h = 0x9E3779B97F4A7C15ull ^ s.n;
    for (int i = 0; i < 4; i++) {
        size_t off = s.n >= 8 ? (s.n - 8) * (size_t)i / 3 : 0;
        uint64_t w = 0;
        memcpy(&w, s.p + off, s.n >= 8 ? 8 : s.n);
        h = (h ^ w) * 0xff51afd7ed558ccdull;
    }
    return h;
}
// Set on the workers of a batch that already runs one tile per host thread: their tiles' loops stay on the worker.  (Measured:
// with 32 tile workers on 16 cores, a nested parallel_for waited ~400 us per call for helper copies that had been started and
// then descheduled - more than the loops' own work.)
thread_local bool tl_serial_loops = false;
thread_local size_t tl_loop_width = 0;  // threads a loop of this thread may occupy, itself included (0: every core)
// fn(i) for i in [0, count): on the caller alone for short loops, otherwise shared with pool threads in chunks of `grain`
template <class F>
void parallel_for(size_t count, size_t grain, F &&fn) {
    const size_t hw = std::max(1u, std::thread::hardware_concurrency());
    if (count < 2 * grain || hw < 2 || tl_serial_loops) {
        for (size_t i = 0; i < count; i++) fn(i);
        return;
    }
    std::atomic<size_t> next{0};
    const std::function<void()> body = [&] {
        for (;;) {
            const size_t lo = next.fetch_add(grain);
            if (lo >= count) break;
            const size_t hi = std::min(count, lo + grain);
            for (size_t i = lo; i < hi; i++) fn(i);
        }
    };
    const size_t width = tl_loop_width ? std::min(tl_loop_width, hw) : hw;
    if (width < 2) {
        body();
        return;
    }
    HostPool::get().run(std::min(width - 1, (count + grain - 1) / grain - 1), body);
}
// the Params every precompile result carries (testnet.rs:8-14) in sunscreen's bincode layout
void testnet_params(uint8_t out[kParamsBytes]) {
    uint64_t w[6] = {(uint64_t)kN, 3, kModulus[MQ0], kModulus[MQ1], kModulus[MP], kT};
    memcpy(out, w, 48);
    memset(out + 48, 0, 8);
}
}  // namespace

Engine &Engine::get() {
    static Engine *e = new Engine();
    return *e;
}
void Engine::set_thread_serial_loops(bool on) { tl_serial_loops = on; }
void Engine::set_thread_loop_width(size_t threads) { tl_loop_width = threads; }

Engine::Engine() {
    HostContext::get();
    n_devices_ = device_count();
    if (n_devices_ <= 0)
        throw std::runtime_error("fhe_b200: no CUDA device visible; this library has no CPU fallback");
    size_t max_dev = env_size("FHE_B200_MAX_DEVICES", (size_t)n_devices_);
    if ((size_t)n_devices_ > max_dev) n_devices_ = (int)max_dev;
    tile_ops_ = env_size("FHE_B200_TILE_OPS", 16);
    if (tile_ops_ < 1) tile_ops_ = 1;
    chunk_ops_ = env_size("FHE_B200_CHUNK_OPS", 4096);
    // byte-surface devices: FHE_B200_DEVICES="0,3" restricts single calls and batches to those GPUs (default: all).
    // Under a one-process-per-GPU launcher each rank sets it to its own device.
    if (const char *v = getenv("FHE_B200_DEVICES")) {
        for (const char *p = v; *p;) {
            char *end = nullptr;
            long d = strtol(p, &end, 10);
            if (end == p) break;
            if (d >= 0 && d < n_devices_) lane_devices_.push_back((int)d);
            p = (*end == ',') ? end + 1 : end;
        }
    }
    if (lane_devices_.empty())
        for (int d = 0; d < n_devices_; d++) lane_devices_.push_back(d);
}

// Lanes (stream + pinned staging + device buffers for one in-flight call) are created on the first byte-surface call,
// so device-resident users never pay for them.  lane_mu_ held.
void Engine::create_lanes() {
    const size_t lanes_per_dev = env_size("FHE_B200_LANES", 32);
    for (int d : lane_devices_) {
        device_context(d);
        for (size_t i = 0; i < lanes_per_dev; i++) {
            std::unique_ptr<Lane> l(new Lane());
            l->device = d;
            l->d_prefix = ct_prefix(d);
            cuda_throw(cudaStreamCreateWithFlags(&l->stream, cudaStreamNonBlocking), "cudaStreamCreate");
            ensure_capacity(l.get(), 1);
            lanes_.push_back(std::move(l));
        }
    }
}

void Engine::drop_graphs(Lane *l) {
    for (auto &g : l->graphs) cudaGraphExecDestroy(g.exec);
    l->graphs.clear();
}

// (re)allocates the lane's staging for `cap` calls; the lane is held by the caller and its stream is idle
void Engine::ensure_capacity(Lane *l, size_t cap) {
    if (l->cap >= cap) return;
    drop_graphs(l);
    cudaFreeHost(l->h_a), cudaFreeHost(l->h_b), cudaFreeHost(l->h_out), cudaFreeHost(l->h_plain);
    cudaFreeHost(l->h_rk_ptrs), cudaFreeHost(l->h_rk_index);
    cudaFree(l->d_a), cudaFree(l->d_b), cudaFree(l->d_out), cudaFree(l->d_plain), cudaFree(l->d_scratch);
    cudaFree(l->d_rk_ptrs), cudaFree(l->d_rk_index);
    l->cap = 0;
    const size_t ct = cap * kCtWords * 8;
    cuda_throw(cudaMallocHost((void **)&l->h_a, ct), "cudaMallocHost");
    cuda_throw(cudaMallocHost((void **)&l->h_b, ct), "cudaMallocHost");
    cuda_throw(cudaMallocHost((void **)&l->h_out, ct), "cudaMallocHost");
    cuda_throw(cudaMallocHost((void **)&l->h_plain, cap * kN * 2), "cudaMallocHost");
    cuda_throw(cudaMalloc((void **)&l->d_a, ct), "cudaMalloc");
    cuda_throw(cudaMalloc((void **)&l->d_b, ct), "cudaMalloc");
    cuda_throw(cudaMalloc((void **)&l->d_out, ct), "cudaMalloc");
    cuda_throw(cudaMalloc((void **)&l->d_plain, cap * kN * 2), "cudaMalloc");
    cuda_throw(cudaMalloc((void **)&l->d_scratch, cap * kScratchLimbsPerOp * kN * 8), "cudaMalloc");
    cuda_throw(cudaMallocHost((void **)&l->h_rk_ptrs, cap * sizeof(uint64_t *)), "cudaMallocHost");
    cuda_throw(cudaMallocHost((void **)&l->h_rk_index, cap * sizeof(int32_t)), "cudaMallocHost");
    cuda_throw(cudaMalloc((void **)&l->d_rk_ptrs, cap * sizeof(uint64_t *)), "cudaMalloc");
    cuda_throw(cudaMalloc((void **)&l->d_rk_index, cap * sizeof(int32_t)), "cudaMalloc");
    l->cap = cap;
}

// device codec buffers for lane->cap calls (two ciphertext operands each)
void Engine::ensure_codec(Lane *l) {
    if (l->codec_cap >= l->cap) return;
    drop_graphs(l);
    cudaFreeHost(l->h_frames), cudaFreeHost(l->h_payloads), cudaFreeHost(l->h_outframes), cudaFreeHost(l->h_jobs), cudaFreeHost(l->h_status);
    cudaFree(l->d_frames), cudaFree(l->d_payloads), cudaFree(l->d_outframes), cudaFree(l->d_jobs), cudaFree(l->d_status), cudaFree(l->d_work);
    l->codec_cap = 0;
    const size_t cap = l->cap, ops = 2 * cap;
    cuda_throw(cudaMallocHost((void **)&l->h_frames, ops * kFrameSlotBytes), "cudaMallocHost");
    cuda_throw(cudaMallocHost((void **)&l->h_payloads, ops * kPayloadStride), "cudaMallocHost");
    cuda_throw(cudaMallocHost((void **)&l->h_outframes, cap * kPackedFrameStride), "cudaMallocHost");
    cuda_throw(cudaMallocHost((void **)&l->h_jobs, ops * sizeof(CodecJob)), "cudaMallocHost");
    cuda_throw(cudaMallocHost((void **)&l->h_status, 3 * cap * sizeof(int32_t)), "cudaMallocHost");
    cuda_throw(cudaMalloc((void **)&l->d_frames, ops * kFrameSlotBytes), "cudaMalloc");
    cuda_throw(cudaMalloc((void **)&l->d_payloads, ops * kPayloadStride), "cudaMalloc");
    cuda_throw(cudaMalloc((void **)&l->d_outframes, cap * kPackedFrameStride), "cudaMalloc");
    cuda_throw(cudaMalloc((void **)&l->d_jobs, ops * sizeof(CodecJob)), "cudaMalloc");
    cuda_throw(cudaMalloc((void **)&l->d_status, 3 * cap * sizeof(int32_t)), "cudaMalloc");
    cuda_throw(cudaMalloc(&l->d_work, ops * codec_work_bytes()), "cudaMalloc");
    l->codec_cap = cap;
}

// the caller has selected `device`
const uint8_t *Engine::ct_prefix(int device) {
    std::lock_guard<std::mutex> lk(prefix_mu_);
    if (d_prefix_.size() < (size_t)n_devices_) d_prefix_.resize((size_t)n_devices_, nullptr);
    uint8_t *&p = d_prefix_[(size_t)device];
    if (!p) {
        uint8_t prefix[kCtPrefixBytes];
        canonical_ct_prefix(prefix);
        cuda_throw(cudaMalloc((void **)&p, kCtPrefixBytes), "cudaMalloc");
        cuda_throw(cudaMemcpy(p, prefix, kCtPrefixBytes, cudaMemcpyHostToDevice), "upload prefix");
    }
    return p;
}

Lane *Engine::acquire_lane() {
    std::unique_lock<std::mutex> lk(lane_mu_);
    if (lanes_.empty()) create_lanes();
    // lowest free lane of the least loaded device: a lone caller keeps reusing lane 0 (warm staging, codec buffers already grown)
    for (;;) {
        Lane *best = nullptr;
        size_t best_busy = ~(size_t)0;
        for (int d : lane_devices_) {
            size_t busy = 0;
            Lane *first_free = nullptr;
            for (auto &l : lanes_) {
                if (l->device != d) continue;
                if (l->busy) busy++;
                else if (!first_free) first_free = l.get();
            }
            if (first_free && busy < best_busy) {
                best = first_free;
                best_busy = busy;
            }
        }
        if (best) {
            best->busy = true;
            return best;
        }
        lane_cv_.wait(lk);
    }
}
void Engine::release_lane(Lane *l) {
    {
        std::lock_guard<std::mutex> lk(lane_mu_);
        l->busy = false;
    }
    lane_cv_.notify_one();
}

// ---------------------------------------------------------------- key cache
KeyPin &KeyPin::operator=(KeyPin &&o) noexcept {
    if (this != &o) {
        release();
        e_ = o.e_;
        k_ = o.k_;
        o.k_ = nullptr;
    }
    return *this;
}
void KeyPin::release() {
    if (k_) e_->unpin_key(k_);
    k_ = nullptr;
}
void Engine::unpin_key(KeyEntry *k) {
    std::lock_guard<std::mutex> lk(key_mu_);
    k->users--;
}

// Content-addressed lookup.  The byte comparison (~400 KB) and a miss's parse run OUTSIDE key_mu_: candidates are pinned
// under the lock (a pinned entry is never evicted and its `bytes` never change), compared without it.
KeyEntry *Engine::find_or_parse_key(Span pk, int32_t *rc) {
    const uint64_t tag = cheap_tag(pk);
    *rc = kOk;
    for (size_t start = 0;;) {
        KeyEntry *cand = nullptr;
        {
            std::lock_guard<std::mutex> lk(key_mu_);
            for (size_t k = start; k < keys_.size(); k++)
                if (keys_[k]->tag == tag && keys_[k]->bytes.size() == pk.n) {
                    cand = keys_[k].get();
                    cand->users++;
                    cand->last_use = ++key_clock_;
                    start = k + 1;
                    break;
                }
        }
        if (!cand) break;
        if (memcmp(cand->bytes.data(), pk.p, pk.n) == 0) return cand;  // pinned
        unpin_key(cand);
    }
    std::unique_ptr<KeyEntry> e(new KeyEntry());
    e->rk.resize(kRkWords);
    e->pk.resize(kPkWords);
    *rc = decode_public_key(pk, e->pk.data(), e->rk.data(), &e->has_relin);
    if (*rc) return nullptr;
    e->bytes.assign(pk.p, pk.p + pk.n);
    e->tag = tag;
    e->d_rk.assign((size_t)n_devices_, nullptr);
    e->d_pk.assign((size_t)n_devices_, nullptr);
    e->users = 1;
    const size_t cap = env_size("FHE_B200_KEY_CACHE", 256);  // a block's users: ~1 MB of host memory each, ~0.6 MB per device

    std::lock_guard<std::mutex> lk(key_mu_);
    for (auto &o : keys_)  // another thread may have inserted the same key meanwhile
        if (o->tag == tag && o->bytes == e->bytes) {
            o->users++;
            o->last_use = ++key_clock_;
            return o.get();
        }
    if (keys_.size() >= cap) {  // evict the least recently used entry nobody is using; if all are pinned, grow
        long victim = -1;
        for (size_t i = 0; i < keys_.size(); i++)
            if (keys_[i]->users == 0 && (victim < 0 || keys_[i]->last_use < keys_[(size_t)victim]->last_use)) victim = (long)i;
        if (victim >= 0) {
            int cur = 0;
            cudaGetDevice(&cur);  // the caller has already selected its lane's device: restore it afterwards
            for (int d = 0; d < n_devices_; d++) {
                uint64_t *ptrs[2] = {keys_[(size_t)victim]->d_rk[(size_t)d], keys_[(size_t)victim]->d_pk[(size_t)d]};
                for (uint64_t *ptr : ptrs)
                    if (ptr) {
                        cudaSetDevice(d);
                        cudaFree(ptr);  // no holder left: every user synchronised its stream before unpinning
                    }
            }
            cudaSetDevice(cur);
            keys_.erase(keys_.begin() + victim);
        }
    }
    e->last_use = ++key_clock_;
    keys_.push_back(std::move(e));
    return keys_.back().get();
}

int32_t Engine::relin_key(Span pk, int device, const uint64_t **d_rk, bool need_relin, KeyPin *pin) {
    int32_t rc = kOk;
    KeyEntry *hit = find_or_parse_key(pk, &rc);  // pinned on success
    if (!hit) return rc;
    KeyPin held(this, hit);
    if (!need_relin) {
        if (d_rk) *d_rk = nullptr;
        return kOk;
    }
    if (!hit->has_relin) return kErrSunscreen;  // sunscreen: relinearization keys required but absent
    {
        std::lock_guard<std::mutex> lk(key_mu_);
        uint64_t *&slot = hit->d_rk[(size_t)device];
        if (!slot) {
            cuda_throw(cudaSetDevice(device), "cudaSetDevice");
            cuda_throw(cudaMalloc((void **)&slot, kRkWords * 8), "cudaMalloc(rk)");
            cuda_throw(cudaMemcpy(slot, hit->rk.data(), kRkWords * 8, cudaMemcpyHostToDevice), "upload rk");
        }
        *d_rk = slot;
    }
    *pin = std::move(held);
    return kOk;
}

int32_t Engine::public_key(Span pk, int device, const uint64_t **d_pk, KeyPin *pin) {
    int32_t rc = kOk;
    KeyEntry *hit = find_or_parse_key(pk, &rc);  // pinned on success
    if (!hit) return rc;
    KeyPin held(this, hit);
    {
        std::lock_guard<std::mutex> lk(key_mu_);
        uint64_t *&slot = hit->d_pk[(size_t)device];
        if (!slot) {
            cuda_throw(cudaSetDevice(device), "cudaSetDevice");
            cuda_throw(cudaMalloc((void **)&slot, kPkWords * 8), "cudaMalloc(pk)");
            cuda_throw(cudaMemcpy(slot, hit->pk.data(), kPkWords * 8, cudaMemcpyHostToDevice), "upload pk");
        }
        *d_pk = slot;
    }
    *pin = std::move(held);
    return kOk;
}

const uint64_t *Engine::network_sk(int device, Span net_pri) {
    std::lock_guard<std::mutex> lk(sk_mu_);
    if (d_net_sk_.size() < (size_t)n_devices_) d_net_sk_.assign((size_t)n_devices_, nullptr);
    uint64_t *&slot = d_net_sk_[(size_t)device];
    if (!slot) {
        std::vector<uint64_t> sk(3 * kN);
        if (decode_private_key(net_pri, sk.data()) != kOk) throw std::runtime_error("fhe_b200: embedded network private key is corrupt");
        cuda_throw(cudaSetDevice(device), "cudaSetDevice");
        cuda_throw(cudaMalloc((void **)&slot, sk.size() * 8), "cudaMalloc(sk)");
        cuda_throw(cudaMemcpy(slot, sk.data(), sk.size() * 8, cudaMemcpyHostToDevice), "upload sk");
    }
    return slot;
}

// ---------------------------------------------------------------- scratch arenas
// One arena per (device, stream): two callers on different streams of one GPU never share scratch, and work already
// enqueued on a stream keeps its arena until that stream has drained (a regrow or an eviction synchronises the owning stream
// first).  A lease pins the arena while its holder is still enqueueing; at most FHE_B200_SCRATCH_ARENAS (default 4) idle arenas
// stay allocated per device (a 4,096-op arena is 7 GB).
Engine::StreamState *Engine::lease_scratch(int device, cudaStream_t s, size_t ops) {
    std::unique_lock<std::mutex> lk(arena_mu_);
    StreamState *st = nullptr;
    for (auto &x : stream_states_)
        if (x->device == device && x->stream == s) st = x.get();
    if (!st) {
        const size_t cap = env_size("FHE_B200_SCRATCH_ARENAS", 4);
        for (;;) {  // evict idle arenas of this device, least recently used first
            size_t have = 0;
            long victim = -1;
            for (size_t i = 0; i < stream_states_.size(); i++) {
                StreamState &x = *stream_states_[i];
                if (x.device != device) continue;
                have++;
                if (x.users == 0 && (victim < 0 || x.last_use < stream_states_[(size_t)victim]->last_use)) victim = (long)i;
            }
            if (have < cap || victim < 0) break;
            StreamState &v = *stream_states_[(size_t)victim];
            cuda_throw(cudaSetDevice(device), "cudaSetDevice");
            if (cudaStreamSynchronize(v.stream) != cudaSuccess) {  // the caller may have destroyed that stream since
                cudaGetLastError();
                cuda_throw(cudaDeviceSynchronize(), "sync before scratch eviction");
            }
            free_stream_state(v);
            stream_states_.erase(stream_states_.begin() + victim);
        }
        stream_states_.emplace_back(new StreamState());
        st = stream_states_.back().get();
        st->device = device;
        st->stream = s;
    }
    // a regrow waits for other holders on the same stream (two threads driving one stream) and for the stream itself
    arena_cv_.wait(lk, [&] { return st->ops >= ops || st->users == 0; });
    if (st->ops < ops) {
        cuda_throw(cudaSetDevice(device), "cudaSetDevice");
        if (st->p) {
            cuda_throw(cudaStreamSynchronize(s), "sync before scratch regrow");
            cudaFree(st->p);
            st->p = nullptr;
            st->ops = 0;
        }
        cuda_throw(cudaMalloc((void **)&st->p, ops * kScratchLimbsPerOp * kN * 8), "cudaMalloc(scratch)");
        st->ops = ops;
    }
    st->users++;
    st->last_use = ++arena_clock_;
    return st;
}
void Engine::release_scratch(StreamState *st) {
    {
        std::lock_guard<std::mutex> lk(arena_mu_);
        st->users--;
    }
    arena_cv_.notify_all();
}
void Engine::free_stream_state(StreamState &v) {
    if (v.p) cudaFree(v.p);
    v.p = nullptr;
}
size_t Engine::set_chunk_ops(long long ops) {
    std::lock_guard<std::mutex> lk(arena_mu_);
    const size_t prev = chunk_ops_;
    if (ops > 0) chunk_ops_ = (size_t)ops;
    return prev;
}
namespace {
struct ScratchLease {
    Engine *e;
    Engine::StreamState *st;
    void (Engine::*rel)(Engine::StreamState *);
    ~ScratchLease() { (e->*rel)(st); }
};
}  // namespace

// ---------------------------------------------------------------- device-resident batched ops
// scratch layout for a chunk of c ops: tens [c][15][N] | c3 [c][6][N] | ks [c][6][N]
cudaEvent_t Engine::take_event() {
    if (!event_pool_.empty()) {
        cudaEvent_t e = event_pool_.back();
        event_pool_.pop_back();
        return e;
    }
    cudaEvent_t e;
    cuda_throw(cudaEventCreate(&e), "cudaEventCreate");
    return e;
}
void Engine::set_kernel_timing(bool on) { timing_ = on; }
void Engine::kernel_timing_report(int device, double ms[kNumTimedKernels], uint64_t launches[kNumTimedKernels]) {
    cuda_throw(cudaSetDevice(device), "cudaSetDevice");
    cuda_throw(cudaDeviceSynchronize(), "sync for timing report");
    std::lock_guard<std::mutex> tlk(timed_mu_);
    for (int k = 0; k < kNumTimedKernels; k++) ms[k] = 0, launches[k] = 0;
    for (auto &t : timed_) {
        float f = 0;
        cuda_throw(cudaEventElapsedTime(&f, t.e0, t.e1), "cudaEventElapsedTime");
        ms[t.kernel] += f;
        launches[t.kernel]++;
        event_pool_.push_back(t.e0);
        event_pool_.push_back(t.e1);
    }
    timed_.clear();
}

// kernel ids (device.py KERNEL_NAMES): 1 k_floor_sk_d, 3 k_relin_finish, 4 k_ext_ntt_d, 5 k_tensor_intt_d, 6 k_digit_ntt,
//             7 k_ks_intt, 8 k_ext_conv_d, 10 k_rk_*_ksd (key preparation), 11 k_digit_ntt_ksd, 14 k_tensor_floor_d,
//             15 k_ks_tail_ksd; 0, 2, 9, 12 and 13 are reserved and never filled
#define TIMED(id, call, what)                                        \
    do {                                                             \
        if (timed) {                                                 \
            std::lock_guard<std::mutex> tlk(timed_mu_);              \
            TimedLaunch tl{id, take_event(), take_event()};          \
            cuda_throw(cudaEventRecord(tl.e0, s), "event record");   \
            cuda_throw(call, what);                                  \
            cuda_throw(cudaEventRecord(tl.e1, s), "event record");   \
            timed_.push_back(tl);                                    \
        } else {                                                     \
            cuda_throw(call, what);                                  \
        }                                                            \
    } while (0)

// Chunks of at least this many ops run the fused tails (k_tensor_floor_d, k_ks_tail_ksd), smaller ones the split tails and the
// key switch on SEAL's key primes.  A fused tail runs three dual words one after the other in one CTA per (output polynomial,
// op): right once its 2 or 3 CTAs per op come close to the 296 resident at a time (2 per SM), three times the critical path
// for a single call or a small tile.
constexpr size_t kFusedTailMinOps = 96;

// BEHZ multiply of c ops: a, b -> m.c3 (size-3 ciphertexts)
void Engine::enqueue_mul(const uint64_t *a, const uint64_t *b, const ScratchMap &m, size_t c, cudaStream_t s, bool timed) {
    TIMED(8, launch_ext_conv(a, b, m.nttbuf, c, s), "ext_conv");
    TIMED(4, launch_ext_ntt(m.nttbuf, c, s), "ext_ntt");
    if (c >= kFusedTailMinOps) {
        TIMED(14, launch_tensor_floor(m.nttbuf, m.c3, c, s), "tensor_floor");
    } else {
        TIMED(5, launch_tensor_intt(m.nttbuf, m.tens, c, s), "tensor_intt");
        TIMED(1, launch_floor_sk(m.tens, m.c3, c, s), "floor_sk");
    }
}
// A prepared dual-base key takes 12 limbs; its preparation passes through 24 limbs of temporaries (coefficient form, lifted).
// A fused chunk runs them through its tensor region (15 limbs per op, dead once c3 exists) in groups of keys that fit.
constexpr size_t kPreparedKeyLimbs = 12, kPrepareTmpLimbs = 24;
static_assert(kPrepareTmpLimbs <= 15 * kFusedTailMinOps, "a fused chunk's tensor region holds the temporaries of one key at least");

// relinearise c size-3 ciphertexts c3 -> out, under rk or (keys) under a key per op
void Engine::enqueue_relin(const uint64_t *c3, const uint64_t *rk, uint64_t *out, const ScratchMap &m, size_t c, cudaStream_t s,
                           bool timed, RelinKeys *keys) {
    if (c >= kFusedTailMinOps) {
        // the whole key switch on the dual base; m.tens (15 limbs per op, dead once c3 exists) holds the lifted key
        const uint64_t *rkd = m.tens + 24 * kN;
        if (!keys) {
            TIMED(10, launch_rk_prepare_ksd(rk, m.tens, s), "rk_prepare_ksd");
        } else {
            if (!keys->ready) {
                size_t group = 15 * c / kPrepareTmpLimbs;
                if (group > kMaxPrepareKeys) group = kMaxPrepareKeys;
                for (size_t k0 = 0; k0 < keys->n_keys; k0 += group) {
                    const size_t g = keys->n_keys - k0 < group ? keys->n_keys - k0 : group;
                    TIMED(10, launch_rk_prepare_keys(nullptr, keys->raw + k0, g, m.tens, keys->prepared + k0 * kPreparedKeyLimbs * kN, s),
                          "rk_prepare_ksd");
                }
                keys->ready = true;
            }
            rkd = keys->prepared;
        }
        TIMED(11, launch_digit_ntt_ksd(c3, m.dig, c, s), "digit_ntt_ksd");
        TIMED(15, launch_ks_tail_ksd(m.dig, rkd, c3, out, c, s, keys ? keys->key_index : nullptr), "ks_tail_ksd");
    } else {
        TIMED(6, launch_digit_ntt(c3, m.dig, c, s), "digit_ntt");
        TIMED(7, launch_ks_intt_keyed(m.dig, rk, keys ? keys->raw : nullptr, keys ? keys->key_index : nullptr, m.ks, c, s), "ks_intt");
        TIMED(3, launch_relin_finish(c3, m.ks, out, c, s), "relin_finish");
    }
}

void Engine::mul_relin(int device, const uint64_t *a, const uint64_t *b, const uint64_t *rk, uint64_t *out, size_t n,
                       cudaStream_t s) {
    if (n == 0) return;
    device_context(device);
    const size_t chunk = chunk_ops_ < n ? chunk_ops_ : n;
    ScratchLease lease{this, lease_scratch(device, s, chunk), &Engine::release_scratch};
    ScratchMap m(lease.st->p, chunk);
    for (size_t off = 0; off < n; off += chunk) {
        const size_t c = n - off < chunk ? n - off : chunk;
        enqueue_mul(a + off * kCtWords, b + off * kCtWords, m, c, s, timing_);
        enqueue_relin(m.c3, rk, out + off * kCtWords, m, c, s, timing_);
    }
}
void Engine::multiply(int device, const uint64_t *a, const uint64_t *b, uint64_t *out3, size_t n, cudaStream_t s) {
    if (n == 0) return;
    device_context(device);
    const size_t chunk = chunk_ops_ < n ? chunk_ops_ : n;
    ScratchLease lease{this, lease_scratch(device, s, chunk), &Engine::release_scratch};
    ScratchMap m(lease.st->p, chunk);
    for (size_t off = 0; off < n; off += chunk) {
        const size_t c = n - off < chunk ? n - off : chunk;
        ScratchMap mm = m;
        mm.c3 = out3 + off * 6 * kN;
        enqueue_mul(a + off * kCtWords, b + off * kCtWords, mm, c, s, false);
    }
}
void Engine::relinearize(int device, const uint64_t *c3, const uint64_t *rk, uint64_t *out, size_t n, cudaStream_t s) {
    if (n == 0) return;
    device_context(device);
    const size_t chunk = chunk_ops_ < n ? chunk_ops_ : n;
    ScratchLease lease{this, lease_scratch(device, s, chunk), &Engine::release_scratch};
    ScratchMap m(lease.st->p, chunk);
    for (size_t off = 0; off < n; off += chunk) {
        const size_t c = n - off < chunk ? n - off : chunk;
        enqueue_relin(c3 + off * 6 * kN, rk, out + off * kCtWords, m, c, s, false);
    }
}

void Engine::mul_relin_keyed(int device, const uint64_t *a, const uint64_t *b, const uint64_t *rks, size_t n_keys,
                             const int32_t *key_index, uint64_t *out, size_t n, cudaStream_t s) {
    keyed_chunks(device, a, b, nullptr, rks, n_keys, key_index, out, n, s);
}
void Engine::relinearize_keyed(int device, const uint64_t *c3, const uint64_t *rks, size_t n_keys, const int32_t *key_index,
                               uint64_t *out, size_t n, cudaStream_t s) {
    keyed_chunks(device, nullptr, nullptr, c3, rks, n_keys, key_index, out, n, s);
}
// The arena holds the chunk's scratch, then the K prepared keys (only when full chunks run the fused tails) and the table of the
// K key pointers; the keys are prepared once, by the first fused chunk, and every chunk may use any of them.
void Engine::keyed_chunks(int device, const uint64_t *a, const uint64_t *b, const uint64_t *c3, const uint64_t *rks, size_t n_keys,
                          const int32_t *key_index, uint64_t *out, size_t n, cudaStream_t s) {
    if (n == 0) return;
    device_context(device);
    const size_t chunk = chunk_ops_ < n ? chunk_ops_ : n;
    const size_t prepared_limbs = chunk >= kFusedTailMinOps ? n_keys * kPreparedKeyLimbs : 0;
    const size_t table_limbs = (n_keys * sizeof(uint64_t *) + kN * 8 - 1) / (kN * 8);
    const size_t extra_ops = (prepared_limbs + table_limbs + kScratchLimbsPerOp - 1) / kScratchLimbsPerOp;
    ScratchLease lease{this, lease_scratch(device, s, chunk + extra_ops), &Engine::release_scratch};
    ScratchMap m(lease.st->p, chunk);
    RelinKeys keys;
    keys.n_keys = n_keys;
    keys.prepared = lease.st->p + chunk * kScratchLimbsPerOp * kN;
    const uint64_t **table = reinterpret_cast<const uint64_t **>(keys.prepared + prepared_limbs * kN);
    keys.raw = table;
    cuda_throw(launch_key_table(rks, kRkWords, n_keys, table, s), "key_table");
    for (size_t off = 0; off < n; off += chunk) {
        const size_t c = n - off < chunk ? n - off : chunk;
        keys.key_index = key_index + off;
        if (a) {
            enqueue_mul(a + off * kCtWords, b + off * kCtWords, m, c, s, timing_);
            enqueue_relin(m.c3, nullptr, out + off * kCtWords, m, c, s, timing_, &keys);
        } else {
            enqueue_relin(c3 + off * 6 * kN, nullptr, out + off * kCtWords, m, c, s, false, &keys);
        }
    }
}

// ---------------------------------------------------------------- host-buffer batch (H2D | kernels | D2H overlapped)
// Chunk schedule of the host pipelines: full chunks in the middle, a short first one (the kernels start after 0.5 ms of copies
// instead of 1.3) and a short last one (less to drain), both of kFusedTailMinOps ops or more where n allows.  For
// kFusedTailMinOps < n < 2 kFusedTailMinOps the remainder after the first chunk is shorter and runs the split tails (n = 150:
// 96 fused + 54 split).  With a pipeline chunk of 96 ops or fewer every chunk runs them, and with one just above 96 the
// next-to-last chunk can be short (97 on 300 ops: 96 / 97 / 11 / 96).  tests/test_edge_parity.py pins these schedules.
// A function of (off, n, chunk) only: every loop over the same batch sees the same chunks.
static size_t pipe_chunk(size_t off, size_t n, size_t chunk) {
    const size_t rem = n - off, edge = kFusedTailMinOps;
    if (chunk <= edge || rem <= edge) return rem < chunk ? rem : chunk;
    if (off == 0) return edge;
    if (rem <= chunk) return rem > 2 * edge ? rem - edge : rem;
    if (rem <= chunk + edge) return rem - edge;
    return chunk;
}

Engine::HostPipe &Engine::host_pipe(int device, const uint64_t *rk, std::unique_lock<std::mutex> &lk) {
    {
        std::lock_guard<std::mutex> g(arena_mu_);
        if (pipes_.size() < (size_t)n_devices_) pipes_.resize((size_t)n_devices_);
        if (!pipes_[(size_t)device]) pipes_[(size_t)device].reset(new HostPipe());
    }
    HostPipe &P = *pipes_[(size_t)device];
    lk = std::unique_lock<std::mutex>(P.mu);
    if (!P.chunk) P.chunk = env_size("FHE_B200_PIPE_CHUNK_OPS", 256);  // (sweep r2w: frames 282 k ops/s at 256 against 260 k at 128; limb arrays equal within noise)
    if (!P.d_rk) cuda_throw(cudaMalloc((void **)&P.d_rk, kRkWords * 8), "cudaMalloc(rk)");
    for (auto &sl : P.slot) {
        if (!sl.stream) cuda_throw(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking), "cudaStreamCreate");
        if (!sl.d_a) {
            cuda_throw(cudaMalloc((void **)&sl.d_a, P.chunk * kCtWords * 8), "cudaMalloc");
            cuda_throw(cudaMalloc((void **)&sl.d_b, P.chunk * kCtWords * 8), "cudaMalloc");
            cuda_throw(cudaMalloc((void **)&sl.d_out, P.chunk * kCtWords * 8), "cudaMalloc");
            cuda_throw(cudaMalloc((void **)&sl.d_scratch, P.chunk * kScratchLimbsPerOp * kN * 8), "cudaMalloc");
        }
    }
    cuda_throw(cudaMemcpyAsync(P.d_rk, rk, kRkWords * 8, cudaMemcpyHostToDevice, P.slot[0].stream), "H2D rk");
    cuda_throw(cudaStreamSynchronize(P.slot[0].stream), "sync rk");
    return P;
}

void Engine::mul_relin_host(int device, const uint64_t *a, const uint64_t *b, const uint64_t *rk, uint64_t *out, size_t n) {
    device_context(device);
    std::unique_lock<std::mutex> lk;
    HostPipe &P = host_pipe(device, rk, lk);
    size_t i = 0;
    for (size_t off = 0, c = 0; off < n; off += c, i++) {
        c = pipe_chunk(off, n, P.chunk);
        PipeSlot &sl = P.slot[i % kPipeSlots];
        cudaStream_t s = sl.stream;
        cuda_throw(cudaMemcpyAsync(sl.d_a, a + off * kCtWords, c * kCtWords * 8, cudaMemcpyHostToDevice, s), "H2D a");
        cuda_throw(cudaMemcpyAsync(sl.d_b, b + off * kCtWords, c * kCtWords * 8, cudaMemcpyHostToDevice, s), "H2D b");
        ScratchMap m(sl.d_scratch, P.chunk);
        enqueue_mul(sl.d_a, sl.d_b, m, c, s, false);
        enqueue_relin(m.c3, P.d_rk, sl.d_out, m, c, s, false);
        cuda_throw(cudaMemcpyAsync(out + off * kCtWords, sl.d_out, c * kCtWords * 8, cudaMemcpyDeviceToHost, s), "D2H out");
    }
    for (auto &sl : P.slot) cuda_throw(cudaStreamSynchronize(sl.stream), "pipe sync");
}

// ---------------------------------------------------------------- serialized operands (structured frames), pipelined like the above
// Operand i of an array is the zstd frame at f + i * stride (the body of a ciphertext this library serialized: 82,054 bytes,
// codec_kernels.h).  Frames are copied as they are (5 bytes per residue instead of 8 over PCIe), validated and unpacked on the
// GPU, and the result is written as a frame on the GPU: fout + i * kPackedFrameStride.  status[i]: 0 done, 1 an operand is not a
// structured frame (or fails the range checks) - result undefined, use the byte surface -, 2 the result needs the generic writer.
void Engine::mul_relin_frames(int device, const uint8_t *fa, const uint8_t *fb, size_t stride, const uint64_t *rk, uint8_t *fout,
                              size_t n, int32_t *status) {
    if (stride < kPackedFrameBytes) throw std::runtime_error("mul_relin_frames: stride smaller than a structured frame");
    device_context(device);
    const uint8_t *prefix = ct_prefix(device);
    std::unique_lock<std::mutex> lk;
    HostPipe &P = host_pipe(device, rk, lk);
    const size_t region = P.chunk * stride;  // one operand array of a chunk
    for (auto &sl : P.slot) {
        if (sl.frame_stride != stride) {  // staging [pad | a frames | pad | b frames | pad], jobs interleaved a0 b0 a1 b1 ...
            cudaFree(sl.d_frames), cudaFree(sl.d_outframes), cudaFree(sl.d_jobs), cudaFree(sl.d_status);
            cuda_throw(cudaMalloc((void **)&sl.d_frames, 2 * region + 3 * kFramePad), "cudaMalloc");
            cuda_throw(cudaMemset(sl.d_frames, 0, 2 * region + 3 * kFramePad), "cudaMemset");
            cuda_throw(cudaMalloc((void **)&sl.d_outframes, P.chunk * kPackedFrameStride), "cudaMalloc");
            cuda_throw(cudaMalloc((void **)&sl.d_jobs, 2 * P.chunk * sizeof(CodecJob)), "cudaMalloc");
            cuda_throw(cudaMalloc((void **)&sl.d_status, 3 * P.chunk * sizeof(int32_t)), "cudaMalloc");
            std::vector<CodecJob> jobs(2 * P.chunk);
            for (size_t i = 0; i < P.chunk; i++) {
                jobs[2 * i] = CodecJob{kFramePad + i * stride, (uint32_t)kPackedFrameBytes, kJobPacked, (int32_t)i, 0};
                jobs[2 * i + 1] = CodecJob{2 * kFramePad + region + i * stride, (uint32_t)kPackedFrameBytes, kJobPacked, (int32_t)i, 1};
            }
            cuda_throw(cudaMemcpy(sl.d_jobs, jobs.data(), jobs.size() * sizeof(CodecJob), cudaMemcpyHostToDevice), "upload jobs");
            sl.frame_stride = stride;
        }
    }
    if (P.h_status_cap < 3 * n) {
        if (P.h_status) cudaFreeHost(P.h_status);
        cuda_throw(cudaMallocHost((void **)&P.h_status, 3 * n * sizeof(int32_t)), "cudaMallocHost");
        P.h_status_cap = 3 * n;
    }
    size_t k = 0;
    for (size_t off = 0, c = 0; off < n; off += c, k++) {
        c = pipe_chunk(off, n, P.chunk);
        PipeSlot &sl = P.slot[k % kPipeSlots];
        cudaStream_t s = sl.stream;
        // the last frame of an array may end before its stride does: never read past fa / fb + (n-1) * stride + frame
        const size_t bytes = (c - 1) * stride + kPackedFrameBytes;
        cuda_throw(cudaMemcpyAsync(sl.d_frames + kFramePad, fa + off * stride, bytes, cudaMemcpyHostToDevice, s), "H2D frames a");
        cuda_throw(cudaMemcpyAsync(sl.d_frames + 2 * kFramePad + region, fb + off * stride, bytes, cudaMemcpyHostToDevice, s), "H2D frames b");
        cuda_throw(launch_codec_inflate(sl.d_frames, nullptr, sl.d_jobs, sl.d_status, nullptr, prefix, sl.d_a, sl.d_b, (int)(2 * c), false,
                                        true, false, s),
                   "frame unpack");
        ScratchMap m(sl.d_scratch, P.chunk);
        enqueue_mul(sl.d_a, sl.d_b, m, c, s, false);
        enqueue_relin(m.c3, P.d_rk, sl.d_out, m, c, s, false);
        cuda_throw(launch_codec_pack(sl.d_out, sl.d_outframes, sl.d_status + 2 * P.chunk, prefix, (int)c, s), "frame pack");
        cuda_throw(cudaMemcpyAsync(fout + off * kPackedFrameStride, sl.d_outframes, (c - 1) * kPackedFrameStride + kPackedFrameBytes,
                                   cudaMemcpyDeviceToHost, s),
                   "D2H frames");
        cuda_throw(cudaMemcpyAsync(P.h_status + 3 * off, sl.d_status, 2 * c * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H status");
        cuda_throw(cudaMemcpyAsync(P.h_status + 3 * off + 2 * c, sl.d_status + 2 * P.chunk, c * sizeof(int32_t), cudaMemcpyDeviceToHost, s),
                   "D2H flags");
    }
    for (auto &sl : P.slot) cuda_throw(cudaStreamSynchronize(sl.stream), "pipe sync");
    if (status) {
        for (size_t off = 0, c = 0; off < n; off += c) {
            c = pipe_chunk(off, n, P.chunk);
            const int32_t *st = P.h_status + 3 * off;
            for (size_t i = 0; i < c; i++) {
                const bool ok = st[2 * i] != kJobFallback && st[2 * i + 1] != kJobFallback;  // the unpack kernel only flags failures
                status[off + i] = !ok ? 1 : (st[2 * c + i] ? 2 : 0);
            }
        }
    }
}

// ---------------------------------------------------------------- serialized <-> device-resident ciphertexts
Engine::XferPipe &Engine::xfer_pipe(int device, size_t n, size_t slot_bytes) {
    {
        std::lock_guard<std::mutex> lk(arena_mu_);
        if (xfers_.size() < (size_t)n_devices_) xfers_.resize((size_t)n_devices_);
        if (!xfers_[(size_t)device]) xfers_[(size_t)device].reset(new XferPipe());
    }
    XferPipe &X = *xfers_[(size_t)device];
    for (auto &sl : X.slot) {
        if (!sl.stream) {
            cuda_throw(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking), "cudaStreamCreate");
            cuda_throw(cudaMalloc((void **)&sl.d_jobs, kXferChunk * sizeof(CodecJob)), "cudaMalloc");
            cuda_throw(cudaMallocHost((void **)&sl.h_jobs, kXferChunk * sizeof(CodecJob)), "cudaMallocHost");
            cuda_throw(cudaMalloc((void **)&sl.d_status, kXferChunk * sizeof(int32_t)), "cudaMalloc");
        }
        if (sl.d_frames_bytes < slot_bytes) {
            cuda_throw(cudaStreamSynchronize(sl.stream), "sync before staging regrow");
            cudaFree(sl.d_frames);
            cuda_throw(cudaMalloc((void **)&sl.d_frames, slot_bytes), "cudaMalloc");
            cuda_throw(cudaMemset(sl.d_frames, 0, slot_bytes), "cudaMemset");
            sl.d_frames_bytes = slot_bytes;
        }
    }
    if (X.h_status_cap < n) {
        if (X.h_status) cudaFreeHost(X.h_status);
        cuda_throw(cudaMallocHost((void **)&X.h_status, n * sizeof(int32_t)), "cudaMallocHost");
        X.h_status_cap = n;
    }
    return X;
}

// frames (host, `stride` apart) -> d_words [n][2][2][N] on `device`.  status[i]: 0 ok, 1 not a structured frame or a residue out
// of range (the words of that ciphertext are then undefined).
void Engine::upload_frames(int device, const uint8_t *frames, size_t stride, size_t n, uint64_t *d_words, int32_t *status) {
    if (n == 0) return;
    if (stride < kPackedFrameBytes) throw std::runtime_error("upload_frames: stride smaller than a structured frame");
    device_context(device);
    const uint8_t *prefix = ct_prefix(device);
    XferPipe &X = xfer_pipe(device, n, kXferChunk * stride + 2 * kFramePad);
    std::lock_guard<std::mutex> lk(X.mu);
    size_t k = 0;
    for (size_t off = 0; off < n; off += kXferChunk, k++) {
        const size_t c = std::min(kXferChunk, n - off);
        XferSlot &sl = X.slot[k & 1];
        cudaStream_t s = sl.stream;
        if (k >= 2) cuda_throw(cudaStreamSynchronize(s), "slot sync");  // h_jobs of this slot are free again
        for (size_t i = 0; i < c; i++) sl.h_jobs[i] = CodecJob{kFramePad + i * stride, (uint32_t)kPackedFrameBytes, kJobPacked, (int32_t)i, 0};
        cuda_throw(cudaMemcpyAsync(sl.d_jobs, sl.h_jobs, c * sizeof(CodecJob), cudaMemcpyHostToDevice, s), "H2D jobs");
        cuda_throw(cudaMemcpyAsync(sl.d_frames + kFramePad, frames + off * stride, (c - 1) * stride + kPackedFrameBytes, cudaMemcpyHostToDevice, s),
                   "H2D frames");
        cuda_throw(launch_codec_inflate(sl.d_frames, nullptr, sl.d_jobs, sl.d_status, nullptr, prefix, d_words + off * kCtWords, nullptr,
                                        (int)c, false, true, false, s),
                   "frame unpack");
        cuda_throw(cudaMemcpyAsync(X.h_status + off, sl.d_status, c * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H status");
    }
    for (auto &sl : X.slot) cuda_throw(cudaStreamSynchronize(sl.stream), "xfer sync");
    if (status)
        for (size_t i = 0; i < n; i++) status[i] = X.h_status[i] == kJobFallback ? 1 : 0;
}

// d_words [n][2][2][N] on `device` -> n structured frames (host, kPackedFrameStride apart).  status[i]: 0 ok, 2 the ciphertext is
// constant (transparent) and has no structured frame: serialise it with fhe_b200_write_ciphertext.
void Engine::download_frames(int device, const uint64_t *d_words, size_t n, uint8_t *out_frames, int32_t *status) {
    if (n == 0) return;
    device_context(device);
    const uint8_t *prefix = ct_prefix(device);
    XferPipe &X = xfer_pipe(device, n, kXferChunk * kPackedFrameStride);
    std::lock_guard<std::mutex> lk(X.mu);
    size_t k = 0;
    for (size_t off = 0; off < n; off += kXferChunk, k++) {
        const size_t c = std::min(kXferChunk, n - off);
        XferSlot &sl = X.slot[k & 1];
        cudaStream_t s = sl.stream;
        cuda_throw(launch_codec_pack(d_words + off * kCtWords, sl.d_frames, sl.d_status, prefix, (int)c, s), "frame pack");
        cuda_throw(cudaMemcpyAsync(out_frames + off * kPackedFrameStride, sl.d_frames, (c - 1) * kPackedFrameStride + kPackedFrameBytes,
                                   cudaMemcpyDeviceToHost, s),
                   "D2H frames");
        cuda_throw(cudaMemcpyAsync(X.h_status + off, sl.d_status, c * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H flags");
    }
    for (auto &sl : X.slot) cuda_throw(cudaStreamSynchronize(sl.stream), "xfer sync");
    if (status)
        for (size_t i = 0; i < n; i++) status[i] = X.h_status[i] ? 2 : 0;
}

// ---------------------------------------------------------------- sunscreen Ciphertexts <-> device-resident ciphertexts
void Engine::xfer_host_stage(XferPipe &X, size_t bytes) {
    for (auto &sl : X.slot) {
        if (sl.h_stage_bytes >= bytes) continue;
        cuda_throw(cudaStreamSynchronize(sl.stream), "sync before staging regrow");
        cudaFreeHost(sl.h_stage);
        sl.h_stage = nullptr, sl.h_stage_bytes = 0;
        cuda_throw(cudaMallocHost((void **)&sl.h_stage, bytes), "cudaMallocHost");
        sl.h_stage_bytes = bytes;
    }
}

namespace {
// what a precompile result of `kind` carries besides its words: the kind's data_type, the testnet Params, compr_mode zstd
CipherView result_view(Kind kind) {
    CipherView v;
    v.data_type = data_type_of(kind);
    testnet_params(v.params);
    v.compr_mode = 2;
    return v;
}

// One ciphertext operand as the codec staging sees it: its bincode framing, data_type and SEAL header (a few hundred bytes).
struct Operand {
    Route route = Route::Reject;
    int32_t rc = kOk;   // Reject: the framing's error code
    CipherView view;    // compr_mode: the blob's
    Span blob, frame;   // the SEAL blob; its zstd frame (Zstd, Packed)
};
// The route of ciphertext `ct` as an operand of `kind`.  Which routes take the device path is the caller's choice.
Route classify_operand(Span ct, Kind kind, Operand *op) {
    if ((op->rc = parse_ciphertext_framing(ct, &op->view, &op->blob))) return op->route = Route::Reject;
    uint8_t compr = 0;
    const int cls = data_type_matches(op->view.data_type, kind) ? classify_ciphertext_blob(op->blob, &op->frame, &compr) : -1;
    if (cls < 0) return op->route = Route::Host;
    op->view.compr_mode = compr;
    if (cls == 0) return op->route = Route::Blob;
    if (op->frame.n + 2 * kFramePad > kFrameSlotBytes) return op->route = Route::Host;
    return op->route = cls == 2 ? Route::Packed : Route::Zstd;
}
// Operand `op`, planned as job j of `jobs`, into the pinned staging: a frame copied to frames + its offset, or a payload the
// host inflates into payloads + j * kPayloadStride.  False if the inflate fails.
bool stage_operand(const Operand &op, const CodecJob *jobs, int32_t j, uint8_t *frames, uint8_t *payloads) {
    if (jobs[j].kind == kJobPayload) {
        uint8_t *dst = payloads + (size_t)j * kPayloadStride;
        return op.route == Route::Blob ? inflate_ct_blob(op.blob, dst) : inflate_ct_payload(op.frame, dst);
    }
    memcpy(frames + jobs[j].src_off, op.frame.p, op.frame.n);
    return true;
}
}  // namespace

// Per ciphertext, on the host pool: classify_operand.  Then, per chunk, one job per ciphertext the device path accepts (Blob,
// Zstd, Packed), laid out by plan_codec_jobs, for launch_codec_inflate, which validates the 97-byte prefix and every residue
// and writes d_words.  Staging of a chunk, the same on the host (pinned) and on the device: [frames | payloads], so that one
// copy moves both.  Every other ciphertext -- and every one the device hands back -- is decoded by decode_ciphertext, whose
// code is the status (the device never turns a valid ciphertext into a rejection).
void Engine::upload_ciphertexts(int device, Kind kind, const uint8_t *const *cts, const size_t *lens, size_t n, uint64_t *d_words,
                                int32_t *status) {
    if (n == 0) return;
    device_context(device);
    const uint8_t *prefix = ct_prefix(device);
    const size_t frames_cap = kXferChunk * kFrameSlotBytes, stage_bytes = frames_cap + kXferChunk * kPayloadStride;
    XferPipe &X = xfer_pipe(device, n, stage_bytes);
    std::lock_guard<std::mutex> lk(X.mu);
    for (auto &sl : X.slot) cuda_throw(cudaStreamSynchronize(sl.stream), "xfer sync");  // (idle unless a call before this one threw)
    xfer_host_stage(X, stage_bytes);
    std::vector<Operand> ops(n);
    std::vector<StageOperand> sop(kXferChunk);
    std::vector<int32_t> job(kXferChunk);
    std::vector<int32_t> st(n, 0);
    struct Pending {
        size_t off = 0, c = 0;
        int jobs = 0;
        bool live = false;
    } pend[2];

    // a chunk's results: ciphertexts handed back by the device join the host route; the host decodes, checks and uploads them
    const auto finish = [&](int b) {
        Pending &p = pend[b];
        XferSlot &sl = X.slot[b];
        p.live = false;
        for (int j = 0; j < p.jobs; j++)
            if (X.h_status[p.off + j] == kJobFallback) ops[p.off + (size_t)sl.h_jobs[j].slot].route = Route::Host;
        std::vector<size_t> host;
        for (size_t i = p.off; i < p.off + p.c; i++)
            if (ops[i].route == Route::Host) host.push_back(i);
        if (host.empty()) return;
        std::vector<std::vector<uint64_t>> words(host.size());
        parallel_for(host.size(), 1, [&](size_t h) {
            const size_t i = host[h];
            CipherView v;
            words[h].resize(kCtWords);
            const int32_t rc = decode_ciphertext(Span{cts[i], lens[i]}, &v, words[h].data());
            st[i] = rc ? rc : data_type_matches(v.data_type, kind) ? kOk : kErrSunscreen;
        });
        for (size_t h = 0; h < host.size(); h++)
            if (st[host[h]] == kOk)
                cuda_throw(cudaMemcpyAsync(d_words + host[h] * kCtWords, words[h].data(), kCtWords * 8, cudaMemcpyHostToDevice, sl.stream),
                           "H2D host-decoded ciphertext");
        cuda_throw(cudaStreamSynchronize(sl.stream), "xfer sync");
    };

    size_t k = 0;
    for (size_t off = 0; off < n; off += kXferChunk, k++) {
        const size_t c = std::min(kXferChunk, n - off);
        const int b = (int)(k & 1);
        XferSlot &sl = X.slot[b];
        cudaStream_t s = sl.stream;
        if (pend[b].live) {  // this slot's staging, jobs and status are free again once its previous chunk is done
            cuda_throw(cudaStreamSynchronize(s), "slot sync");
            finish(b);
        }
        // (A) framing, data_type and blob header of every ciphertext of the chunk
        parallel_for(c, 8, [&](size_t t) {
            Operand &o = ops[off + t];
            if (classify_operand(Span{cts[off + t], lens[off + t]}, kind, &o) == Route::Reject) st[off + t] = o.rc;
            sop[t] = StageOperand{o.route, o.frame.n, (int32_t)t, 0};
        });
        // (B) the jobs; (C) frames into the staging as they are, payloads inflated (or copied) into their slots
        const StagePlan plan = plan_codec_jobs(sop.data(), c, sl.h_jobs, job.data());
        const size_t pay_base = (plan.frame_bytes + 255) & ~(size_t)255;
        parallel_for(c, 2, [&](size_t t) {
            if (job[t] >= 0 && !stage_operand(ops[off + t], sl.h_jobs, job[t], sl.h_stage, sl.h_stage + pay_base)) {
                ops[off + t].route = Route::Host;
                sl.h_jobs[job[t]].kind = kJobNone;
            }
        });
        // (D) one copy of the staging, the jobs, the codec kernels straight into d_words, the job status back
        if (plan.jobs) {
            const size_t bytes = plan.payloads ? pay_base + (size_t)plan.payloads * kPayloadStride : plan.frame_bytes;
            if (plan.any_zstd && !sl.d_work) cuda_throw(cudaMalloc(&sl.d_work, kXferChunk * codec_work_bytes()), "cudaMalloc");
            cuda_throw(cudaMemcpyAsync(sl.d_jobs, sl.h_jobs, (size_t)plan.jobs * sizeof(CodecJob), cudaMemcpyHostToDevice, s), "H2D jobs");
            cuda_throw(cudaMemcpyAsync(sl.d_frames, sl.h_stage, bytes, cudaMemcpyHostToDevice, s), "H2D ciphertexts");
            cuda_throw(launch_codec_inflate(sl.d_frames, sl.d_frames + pay_base, sl.d_jobs, sl.d_status, sl.d_work, prefix,
                                            d_words + off * kCtWords, nullptr, plan.jobs, plan.any_zstd, plan.any_packed, plan.payloads > 0, s),
                       "ciphertext unpack");
            cuda_throw(cudaMemcpyAsync(X.h_status + off, sl.d_status, (size_t)plan.jobs * sizeof(int32_t), cudaMemcpyDeviceToHost, s),
                       "D2H status");
        }
        pend[b] = Pending{off, c, plan.jobs, true};
    }
    for (int b = 0; b < 2; b++) {
        const int oldest = (int)((k + (size_t)b) & 1);  // (in chunk order)
        if (!pend[oldest].live) continue;
        cuda_throw(cudaStreamSynchronize(X.slot[oldest].stream), "xfer sync");
        finish(oldest);
    }
    if (status) memcpy(status, st.data(), n * sizeof(int32_t));
}

// Structured writer: k_ct_pack40 writes every row as the complete Ciphertext (the kind's constant envelope, then the frame) and
// one copy per chunk brings the final bytes back; constant (transparent) results take encode_ciphertext, as on the byte surface.
// Default writer (SEAL's own bytes, libzstd level 3 on the host cores): one copy of the words per chunk, encode_ciphertext on
// the host pool.  Either way the host works on chunk k while the device and PCIe work on chunk k + 1.
void Engine::download_ciphertexts(int device, Kind kind, const uint64_t *d_words, size_t n, uint8_t **outputs, int64_t *output_lengths,
                                  int32_t *status, std::string *row_error) {
    if (n == 0) return;
    device_context(device);
    const CipherView view = result_view(kind);
    const bool structured = zstd_writer() == 1;
    const size_t head = wrapped_ciphertext_size(view, kPackedFrameBytes) - kPackedFrameBytes, whole = head + kPackedFrameBytes;
    if (head > (size_t)kPackHeadMax) throw std::runtime_error("download_ciphertexts: data_type too long");
    const size_t row = structured ? (whole + 15) & ~(size_t)15 : kCtWords * 8;
    const uint8_t *prefix = ct_prefix(device);
    XferPipe &X = xfer_pipe(device, n, kXferChunk * row);
    std::lock_guard<std::mutex> lk(X.mu);
    for (auto &sl : X.slot) cuda_throw(cudaStreamSynchronize(sl.stream), "xfer sync");  // (idle unless a call before this one threw)
    xfer_host_stage(X, kXferChunk * row);
    if (structured) {
        std::vector<uint8_t> zero(kPackedFrameBytes, 0), env(whole);
        wrap_ciphertext_blob_to(view, zero.data(), kPackedFrameBytes, env.data());
        if (!X.d_head) cuda_throw(cudaMalloc((void **)&X.d_head, kPackHeadMax), "cudaMalloc");
        cuda_throw(cudaMemcpy(X.d_head, env.data(), head, cudaMemcpyHostToDevice), "upload envelope");
    }
    std::mutex err_mu;
    struct Pending {
        size_t off = 0, c = 0;
        bool live = false;
    } pend[2];
    const auto finish = [&](int b) {
        Pending &p = pend[b];
        XferSlot &sl = X.slot[b];
        p.live = false;
        cuda_throw(cudaStreamSynchronize(sl.stream), "xfer sync");  // the chunk's bytes (or words) and constant flags are here
        std::vector<std::vector<uint64_t>> constant(p.c);           // words of the constant results (structured writer)
        bool any_constant = false;
        if (structured)
            for (size_t t = 0; t < p.c; t++)
                if (X.h_status[p.off + t]) {
                    constant[t].resize(kCtWords);
                    any_constant = true;
                    cuda_throw(cudaMemcpyAsync(constant[t].data(), d_words + (p.off + t) * kCtWords, kCtWords * 8, cudaMemcpyDeviceToHost, sl.stream),
                               "D2H constant result");
                }
        if (any_constant) cuda_throw(cudaStreamSynchronize(sl.stream), "xfer sync");
        parallel_for(p.c, 4, [&](size_t t) {
            const size_t i = p.off + t;
            outputs[i] = nullptr, output_lengths[i] = 0, status[i] = -1;
            try {
                thread_local std::vector<uint8_t> bytes;
                const uint8_t *src = sl.h_stage + t * row;
                size_t len = whole;
                if (!structured || !constant[t].empty()) {
                    encode_ciphertext(view, structured ? constant[t].data() : reinterpret_cast<const uint64_t *>(src), &bytes);
                    src = bytes.data(), len = bytes.size();
                }
                uint8_t *o = (uint8_t *)malloc(len);
                if (!o) throw std::runtime_error("download_ciphertexts: out of host memory");
                memcpy(o, src, len);
                outputs[i] = o, output_lengths[i] = (int64_t)len, status[i] = 0;
            } catch (const std::exception &e) {
                std::lock_guard<std::mutex> g(err_mu);
                if (row_error && row_error->empty()) *row_error = "download_ciphertexts: ciphertext " + std::to_string(i) + ": " + e.what();
            }
        });
    };
    size_t k = 0;
    for (size_t off = 0; off < n; off += kXferChunk, k++) {
        const size_t c = std::min(kXferChunk, n - off);
        const int b = (int)(k & 1);
        XferSlot &sl = X.slot[b];
        cudaStream_t s = sl.stream;
        if (pend[b].live) finish(b);
        if (structured) {
            cuda_throw(launch_codec_pack(d_words + off * kCtWords, sl.d_frames, row, X.d_head, (int)head, sl.d_status, prefix, (int)c, s),
                       "ciphertext pack");
            cuda_throw(cudaMemcpyAsync(sl.h_stage, sl.d_frames, (c - 1) * row + whole, cudaMemcpyDeviceToHost, s), "D2H ciphertexts");
            cuda_throw(cudaMemcpyAsync(X.h_status + off, sl.d_status, c * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H flags");
        } else {
            cuda_throw(cudaMemcpyAsync(sl.h_stage, d_words + off * kCtWords, c * kCtWords * 8, cudaMemcpyDeviceToHost, s), "D2H words");
        }
        pend[b] = Pending{off, c, true};
    }
    for (int b = 0; b < 2; b++) {
        const int oldest = (int)((k + (size_t)b) & 1);
        if (pend[oldest].live) finish(oldest);
    }
}

// ---------------------------------------------------------------- byte surface, one call
namespace {
struct LaneGuard {
    Engine *e;
    Lane *l;
    void (Engine::*rel)(Lane *);
    ~LaneGuard() { (e->*rel)(l); }
};
}  // namespace

namespace {
thread_local CallBreakdown tl_breakdown;
inline double us_since(std::chrono::steady_clock::time_point t0) {
    return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
}
}  // namespace
const CallBreakdown &Engine::last_call_breakdown() { return tl_breakdown; }

int32_t Engine::binary_op(Op op, Shape shape, Kind kind, Span in, std::vector<uint8_t> *out) {
    TileItem it{op, shape, kind, in, {}, 0};
    binary_tile(&it, 1);
    if (it.rc == 0) out->swap(it.out);
    return it.rc;
}

// One call whose inputs are perfectly ordinary (the overwhelmingly common case), arranged for latency: the public-key
// comparison and the inflate of the first operand run on the caller while a pool thread inflates the second operand; payloads
// are validated and unpacked on the GPU and the result frame is written there.  Returns false -- having produced nothing --
// whenever anything deviates; binary_tile's general path then redoes the call and owns every error code.
bool Engine::single_call_fast(Lane *lane, TileItem &it, bool timed, std::chrono::steady_clock::time_point t_start) {
    Span pk, sa, sb;
    if (unpack_binary_operation(it.in, &pk, &sa, &sb)) return false;
    const int nct = it.shape == Shape::CtCt ? 2 : 1;
    const Span cts[2] = {it.shape == Shape::PtCt ? sb : sa, sb};
    Operand ops[2];
    StageOperand sop[2];
    for (int k = 0; k < nct; k++) {
        const Route r = classify_operand(cts[k], it.kind, &ops[k]);
        if (r != Route::Zstd && r != Route::Packed) return false;
        sop[k] = StageOperand{r, ops[k].frame.n, 0, k};
    }
    if (zstd_writer() != 1) return false;
    ensure_codec(lane);
    cudaStream_t s = lane->stream;

    // libzstd frames are inflated here (two never reach kDeviceZstdMinFrames), and a structured frame has one size: the plan,
    // and so every copy below, is fixed for a pair of routes and is replayed as a graph
    int32_t job[2];
    const StagePlan plan = plan_codec_jobs(sop, (size_t)nct, lane->h_jobs, job);
    const bool need_relin = it.op == Op::Mul && it.shape == Shape::CtCt;
    const uint64_t *d_rk = nullptr;
    KeyPin pin;
    int32_t key_rc = kOk;
    bool staged[2] = {true, true};
    std::atomic<int> next{0};
    const std::function<void()> work = [&] {  // tasks: first operand, second operand (ct x ct only), key comparison
        for (int t; (t = next.fetch_add(1)) < 3;) {
            if (t == 2) key_rc = relin_key(pk, lane->device, &d_rk, need_relin, &pin);
            else if (t < nct) staged[t] = stage_operand(ops[t], lane->h_jobs, job[t], lane->h_frames, lane->h_payloads);
        }
    };
    HostPool::get().run((size_t)nct, work);
    if (key_rc != kOk || !staged[0] || !staged[1]) return false;
    if (it.shape != Shape::CtCt && encode_scalar(it.kind, it.shape == Shape::CtPt ? sb : sa, lane->h_plain) != kOk) return false;
    const double t_decode = us_since(t_start);

    int32_t *d_cflag = lane->d_status + nct, *h_cflag = lane->h_status + nct;  // right behind the job status: one copy back
    const auto enqueue = [&](bool ev) {
        if (ev) cudaEventRecord(lane->ev[0], s);
        cuda_throw(cudaMemcpyAsync(lane->d_jobs, lane->h_jobs, (size_t)nct * sizeof(CodecJob), cudaMemcpyHostToDevice, s), "H2D jobs");
        if (plan.frame_bytes)
            cuda_throw(cudaMemcpyAsync(lane->d_frames, lane->h_frames, plan.frame_bytes, cudaMemcpyHostToDevice, s), "H2D frames");
        if (plan.payloads)
            cuda_throw(cudaMemcpyAsync(lane->d_payloads, lane->h_payloads, (size_t)plan.payloads * kPayloadStride, cudaMemcpyHostToDevice, s),
                       "H2D payloads");
        if (it.shape != Shape::CtCt) cuda_throw(cudaMemcpyAsync(lane->d_plain, lane->h_plain, kN * 2, cudaMemcpyHostToDevice, s), "H2D plain");
        if (ev) cudaEventRecord(lane->ev[1], s);
        cuda_throw(launch_codec_inflate(lane->d_frames, lane->d_payloads, lane->d_jobs, lane->d_status, lane->d_work, lane->d_prefix, lane->d_a,
                                        lane->d_b, nct, plan.any_zstd, plan.any_packed, plan.payloads > 0, s),
                   "codec unpack");
        if (it.shape == Shape::CtCt) {
            if (it.op == Op::Mul) {
                ScratchMap m(lane->d_scratch, 1);
                enqueue_mul(lane->d_a, lane->d_b, m, 1, s, false);
                enqueue_relin(m.c3, d_rk, lane->d_out, m, 1, s, false);
            } else {
                cuda_throw(launch_eltwise(lane->d_a, lane->d_b, lane->d_out, 1, it.op == Op::Add ? 0 : 1, s), "eltwise");
            }
        } else if (it.op == Op::Mul) {
            cuda_throw(launch_mul_plain(lane->d_a, lane->d_plain, lane->d_out, 1, s), "mul_plain");
        } else {
            const int mode = it.op == Op::Add ? 0 : (it.shape == Shape::CtPt ? 1 : 3);
            cuda_throw(launch_plain_addsub(lane->d_a, lane->d_plain, lane->d_out, 1, mode, s), "plain_addsub");
        }
        cuda_throw(launch_codec_pack(lane->d_out, lane->d_outframes, d_cflag, lane->d_prefix, 1, s), "codec pack");
        if (ev) cudaEventRecord(lane->ev[2], s);
        cuda_throw(cudaMemcpyAsync(lane->h_outframes, lane->d_outframes, kPackedFrameBytes, cudaMemcpyDeviceToHost, s), "D2H frame");
        cuda_throw(cudaMemcpyAsync(lane->h_status, lane->d_status, (size_t)(nct + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H status");
        if (ev) cudaEventRecord(lane->ev[3], s);
    };
    // every size and pointer above is fixed for a given call shape and pair of routes on this lane (the result frame has a
    // constant size too), so the sequence is replayed as a CUDA graph: ~13 launches and copies become one
    if (!timed) {
        cudaGraphExec_t exec = nullptr;
        for (const auto &g : lane->graphs)
            if (g.op == (int)it.op && g.shape == (int)it.shape && g.route0 == (int)ops[0].route && g.route1 == (int)ops[1].route && g.rk == d_rk) {
                exec = g.exec;
                count_launches(g.launches);
            }
        if (!exec) {
            const uint64_t before = launch_count() + codec_launch_count();
            if (lane->graphs.size() >= 16) drop_graphs(lane);
            cudaGraph_t graph = nullptr;
            cuda_throw(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal), "begin capture");
            try {
                enqueue(false);
            } catch (...) {
                cudaStreamEndCapture(s, &graph);
                if (graph) cudaGraphDestroy(graph);
                throw;
            }
            cuda_throw(cudaStreamEndCapture(s, &graph), "end capture");
            cuda_throw(cudaGraphInstantiate(&exec, graph, 0), "graph instantiate");
            cudaGraphDestroy(graph);
            lane->graphs.push_back(Lane::CallGraph{(int)it.op, (int)it.shape, (int)ops[0].route, (int)ops[1].route, d_rk, exec,
                                                   launch_count() + codec_launch_count() - before});
        }
        cuda_throw(cudaGraphLaunch(exec, s), "graph launch");
    } else {
        enqueue(timed);
    }
    cuda_throw(cudaStreamSynchronize(s), "stream sync");
    const double t_device = us_since(t_start);
    for (int k = 0; k < nct; k++)
        if (lane->h_status[k] == kJobFallback) return false;
    if (h_cflag[0]) {  // constant result (a transparent ciphertext): the host writer's libzstd path
        cuda_throw(cudaMemcpyAsync(lane->h_out, lane->d_out, kCtWords * 8, cudaMemcpyDeviceToHost, s), "D2H");
        cuda_throw(cudaStreamSynchronize(s), "stream sync");
        it.rc = encode_ciphertext(ops[0].view, lane->h_out, &it.out);
    } else {
        wrap_ciphertext_blob(ops[0].view, lane->h_outframes, kPackedFrameBytes, &it.out);
        it.rc = kOk;
    }
    if (timed) {
        CallBreakdown &b = tl_breakdown;
        float ms[3] = {0, 0, 0};
        for (int k = 0; k < 3; k++) cudaEventElapsedTime(&ms[k], lane->ev[k], lane->ev[k + 1]);
        b.unpack_key_us = 0;  // the key comparison overlaps the inflates on this path
        b.decode_us = t_decode;
        b.h2d_us = ms[0] * 1e3;
        b.kernels_us = ms[1] * 1e3;
        b.d2h_us = ms[2] * 1e3;
        b.total_us = us_since(t_start);
        b.encode_us = b.total_us - t_device;
    }
    return true;
}

void Engine::binary_tile(TileItem *items, size_t cnt) {
    if (cnt == 0) return;
    const bool timed = call_timing_.load(std::memory_order_relaxed);
    const auto t_start = std::chrono::steady_clock::now();
    Lane *lane = acquire_lane();
    LaneGuard guard{this, lane, &Engine::release_lane};
    cuda_throw(cudaSetDevice(lane->device), "cudaSetDevice");
    ensure_capacity(lane, cnt);
    cudaStream_t s = lane->stream;
    if (timed && !lane->ev[0])
        for (auto &e : lane->ev) cuda_throw(cudaEventCreate(&e), "cudaEventCreate");

    if (cnt == 1 && single_call_fast(lane, items[0], timed, t_start)) return;

    // device work classes; ct-ct first so that the second operand array is one prefix of the slots
    enum Cls { kMulCt = 0, kAddCt, kSubCt, kMulPt, kAddPt, kSubCtPt, kSubPtCt };
    struct Prep {
        Span sa, sb;
        const uint64_t *d_rk = nullptr;
        KeyPin pin;
        int32_t key_rc = 0;
        CipherView va;
        int cls = 0;
        bool live = false;
    };
    std::vector<Prep> prep(cnt);
    std::vector<size_t> order;
    order.reserve(cnt);

    // pass 1, reference order (pack.rs:261-263): framing, then the public key (a ~400 KB comparison with the cached key per call:
    // shared with pool threads when the tile is large)
    parallel_for(cnt, 4, [&](size_t i) {
        TileItem &it = items[i];
        Prep &p = prep[i];
        Span pk;
        if ((it.rc = unpack_binary_operation(it.in, &pk, &p.sa, &p.sb))) return;
        const bool need_relin = (it.op == Op::Mul && it.shape == Shape::CtCt);
        int32_t rc = relin_key(pk, lane->device, &p.d_rk, need_relin, &p.pin);
        if (rc == kErrSunscreen && need_relin) {
            // missing relin keys is a runtime (not a decoding) error: operands are still decoded first
        } else if (rc) {
            it.rc = rc;
            return;
        }
        p.key_rc = rc;
        if (it.shape == Shape::CtCt) p.cls = it.op == Op::Mul ? kMulCt : (it.op == Op::Add ? kAddCt : kSubCt);
        else if (it.op == Op::Mul) p.cls = kMulPt;
        else if (it.op == Op::Add) p.cls = kAddPt;
        else p.cls = it.shape == Shape::CtPt ? kSubCtPt : kSubPtCt;
        p.live = true;
    });
    for (size_t i = 0; i < cnt; i++)
        if (prep[i].live) order.push_back(i);
    const double t_unpack = us_since(t_start);
    // one run per class: a pass launches all its ct-ct multiplies as one run, whatever keys they use
    struct Run {
        int cls;
        size_t begin, end;
    };
    // the multiply run's keys: the distinct keys in order of first appearance, and each slot's index into them
    struct RunKeys {
        std::vector<const uint64_t *> keys;
        std::vector<int32_t> index;
        void add(const uint64_t *rk) {
            if (keys.empty() || keys.back() != rk) keys.push_back(rk);  // the class is sorted by key
            index.push_back((int32_t)keys.size() - 1);
        }
    };
    // ops sharing a key sit next to each other: their key reads hit in L2
    const auto by_class = [&](size_t x, size_t y) {
        if (prep[x].cls != prep[y].cls) return prep[x].cls < prep[y].cls;
        return prep[x].cls == kMulCt && prep[x].d_rk < prep[y].d_rk;
    };
    // a tile has at most one key per op, so its prepared keys fit the extension buffer, dead once the tensor product exists
    static_assert(kPreparedKeyLimbs <= 20, "prepared keys (one per op at most) in nttbuf (20 limbs per op)");
    const auto launch_runs = [&](const std::vector<Run> &rs, RunKeys &rk) {
        for (const Run &r : rs) {
            const size_t c = r.end - r.begin;
            const uint64_t *a = lane->d_a + r.begin * kCtWords;
            const uint64_t *b = lane->d_b + r.begin * kCtWords;
            const uint16_t *pl = lane->d_plain + r.begin * kN;
            uint64_t *o = lane->d_out + r.begin * kCtWords;
            switch (r.cls) {
                case kMulCt: {
                    ScratchMap m(lane->d_scratch, c);
                    enqueue_mul(a, b, m, c, s, false);
                    if (rk.keys.size() == 1) {
                        enqueue_relin(m.c3, rk.keys[0], o, m, c, s, false);
                        break;
                    }
                    const size_t k = rk.keys.size();
                    memcpy(lane->h_rk_ptrs, rk.keys.data(), k * sizeof(uint64_t *));
                    memcpy(lane->h_rk_index, rk.index.data(), c * sizeof(int32_t));
                    cuda_throw(cudaMemcpyAsync(lane->d_rk_ptrs, lane->h_rk_ptrs, k * sizeof(uint64_t *), cudaMemcpyHostToDevice, s), "H2D keys");
                    cuda_throw(cudaMemcpyAsync(lane->d_rk_index, lane->h_rk_index, c * sizeof(int32_t), cudaMemcpyHostToDevice, s),
                               "H2D key indices");
                    RelinKeys keys;
                    keys.raw = lane->d_rk_ptrs;
                    keys.n_keys = k;
                    keys.prepared = m.nttbuf;
                    keys.key_index = lane->d_rk_index;
                    enqueue_relin(m.c3, nullptr, o, m, c, s, false, &keys);
                    break;
                }
                case kAddCt: cuda_throw(launch_eltwise(a, b, o, c, 0, s), "eltwise"); break;
                case kSubCt: cuda_throw(launch_eltwise(a, b, o, c, 1, s), "eltwise"); break;
                case kMulPt: cuda_throw(launch_mul_plain(a, pl, o, c, s), "mul_plain"); break;
                // a + b: add_plain; ct - pt: sub_plain; pt - ct: negate(sub_plain(ct, pt))  (SURVEY 3.1)
                case kAddPt: cuda_throw(launch_plain_addsub(a, pl, o, c, 0, s), "plain_addsub"); break;
                case kSubCtPt: cuda_throw(launch_plain_addsub(a, pl, o, c, 1, s), "plain_addsub"); break;
                default: cuda_throw(launch_plain_addsub(a, pl, o, c, 3, s), "plain_addsub"); break;
            }
        }
    };
    std::stable_sort(order.begin(), order.end(), by_class);

    // ---- device codec pass (tiles only): calls whose operands are zstd-mode ciphertexts with clean framing travel as
    // compressed frames; the GPU inflates, validates, computes and packs the result frame.  Whatever is not perfectly
    // ordinary -- and every operand the strict device decoder hands back -- is left for the host pass below, which
    // reproduces the reference's checks and error codes in their order.
    if (cnt >= 2 && !order.empty()) {
        ensure_codec(lane);
        std::vector<Run> runs;
        RunKeys run_keys;
        std::vector<size_t> slot_item, rest;
        const bool pack_on_device = zstd_writer() == 1;
        // (A) per call, in parallel: classify_operand; a call takes the device path when all its operands are Zstd or Packed
        struct Stg {
            bool clean = false;
            int nct = 0;
            Operand ops[2];
            size_t op0 = 0;                // its first operand in the plan: operand c is staged as job[op0 + c]
            std::atomic<bool> bad{false};  // staging failed: the host pass redoes the call
        };
        std::vector<Stg> stg(order.size());
        parallel_for(order.size(), 8, [&](size_t oi) {
            const size_t i = order[oi];
            TileItem &it = items[i];
            Stg &g = stg[oi];
            const Span cts[2] = {it.shape == Shape::PtCt ? prep[i].sb : prep[i].sa, prep[i].sb};
            g.nct = it.shape == Shape::CtCt ? 2 : 1;
            g.clean = prep[i].key_rc == 0;
            for (int k = 0; g.clean && k < g.nct; k++) {
                const Route r = classify_operand(cts[k], it.kind, &g.ops[k]);
                g.clean = r == Route::Zstd || r == Route::Packed;
            }
        });
        // (B) serial: slots, then the jobs of every clean call's operands
        size_t slots = 0, ctct_slots = 0;
        std::vector<size_t> slot_stg;
        std::vector<StageOperand> sop;
        for (size_t oi = 0; oi < order.size(); oi++) {
            const size_t i = order[oi];
            Stg &g = stg[oi];
            Prep &p = prep[i];
            if (!g.clean) {
                rest.push_back(i);
                continue;
            }
            p.va = g.ops[0].view;
            g.op0 = sop.size();
            for (int k = 0; k < g.nct; k++) sop.push_back(StageOperand{g.ops[k].route, g.ops[k].frame.n, (int32_t)slots, k});
            if (p.cls == kMulCt) run_keys.add(p.d_rk);
            if (runs.empty() || runs.back().cls != p.cls) runs.push_back(Run{p.cls, slots, slots});
            runs.back().end = ++slots;
            if (p.cls <= kSubCt) ctct_slots = slots;
            slot_item.push_back(i);
            slot_stg.push_back(oi);
        }
        std::vector<int32_t> job(sop.size());
        const StagePlan plan = plan_codec_jobs(sop.data(), sop.size(), lane->h_jobs, job.data());
        if (slots) {
            // (C) bytes into the pinned staging -- frames as they are, encoded scalars; (C2) the frames cross to the device while
            // the host inflates the libzstd frames of a tile that is too small for the device decoder
            const auto fail_slot = [&](Stg &g) {
                g.bad = true;
                for (int c = 0; c < g.nct; c++) lane->h_jobs[job[g.op0 + c]].kind = kJobNone;  // the kernels skip it; its slot computes on stale data
            };
            parallel_for(slots, 2, [&](size_t k) {
                Stg &g = stg[slot_stg[k]];
                TileItem &it = items[slot_item[k]];
                Prep &p = prep[slot_item[k]];
                for (int c = 0; c < g.nct; c++)
                    if (lane->h_jobs[job[g.op0 + c]].kind != kJobPayload)
                        stage_operand(g.ops[c], lane->h_jobs, job[g.op0 + c], lane->h_frames, lane->h_payloads);
                if (it.shape != Shape::CtCt && encode_scalar(it.kind, it.shape == Shape::CtPt ? p.sb : p.sa, lane->h_plain + k * kN) != kOk)
                    fail_slot(g);
            });
            if (plan.frame_bytes)
                cuda_throw(cudaMemcpyAsync(lane->d_frames, lane->h_frames, plan.frame_bytes, cudaMemcpyHostToDevice, s), "H2D frames");
            cuda_throw(cudaMemcpyAsync(lane->d_jobs, lane->h_jobs, (size_t)plan.jobs * sizeof(CodecJob), cudaMemcpyHostToDevice, s), "H2D jobs");
            if (plan.payloads) {
                std::atomic<bool> any_failed{false};
                parallel_for(slots, 2, [&](size_t k) {
                    Stg &g = stg[slot_stg[k]];
                    if (g.bad) return;
                    for (int c = 0; c < g.nct; c++) {
                        const int32_t j = job[g.op0 + c];
                        if (lane->h_jobs[j].kind == kJobPayload && !stage_operand(g.ops[c], lane->h_jobs, j, lane->h_frames, lane->h_payloads)) {
                            fail_slot(g);
                            any_failed = true;
                            break;
                        }
                    }
                });
                if (any_failed)  // (the first copy of the job list may or may not have seen the cleared kinds: either is fine)
                    cuda_throw(cudaMemcpyAsync(lane->d_jobs, lane->h_jobs, (size_t)plan.jobs * sizeof(CodecJob), cudaMemcpyHostToDevice, s), "H2D jobs");
                cuda_throw(cudaMemcpyAsync(lane->d_payloads, lane->h_payloads, (size_t)plan.payloads * kPayloadStride, cudaMemcpyHostToDevice, s),
                           "H2D payloads");
            }
            if (slots > ctct_slots)
                cuda_throw(cudaMemcpyAsync(lane->d_plain + ctct_slots * kN, lane->h_plain + ctct_slots * kN,
                                           (slots - ctct_slots) * kN * 2, cudaMemcpyHostToDevice, s),
                           "H2D plain");
            cuda_throw(launch_codec_inflate(lane->d_frames, lane->d_payloads, lane->d_jobs, lane->d_status, lane->d_work, lane->d_prefix,
                                            lane->d_a, lane->d_b, plan.jobs, plan.any_zstd, plan.any_packed, plan.payloads > 0, s),
                       "codec inflate");
            launch_runs(runs, run_keys);
            int32_t *d_cflag = lane->d_status + 2 * lane->cap, *h_cflag = lane->h_status + 2 * lane->cap;
            if (pack_on_device) {
                cuda_throw(launch_codec_pack(lane->d_out, lane->d_outframes, d_cflag, lane->d_prefix, (int)slots, s), "codec pack");
                cuda_throw(cudaMemcpyAsync(lane->h_outframes, lane->d_outframes, slots * kPackedFrameStride, cudaMemcpyDeviceToHost, s),
                           "D2H frames");
                cuda_throw(cudaMemcpyAsync(h_cflag, d_cflag, slots * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H flags");
            } else {
                cuda_throw(cudaMemcpyAsync(lane->h_out, lane->d_out, slots * kCtWords * 8, cudaMemcpyDeviceToHost, s), "D2H");
            }
            cuda_throw(cudaMemcpyAsync(lane->h_status, lane->d_status, (size_t)plan.jobs * sizeof(int32_t), cudaMemcpyDeviceToHost, s),
                       "D2H status");
            cuda_throw(cudaStreamSynchronize(s), "stream sync");
            // (D) in parallel: results into their own buffers; calls the device handed back are collected for the host pass
            std::vector<uint8_t> redo(slots, 0);
            parallel_for(slots, 4, [&](size_t k) {
                const size_t i = slot_item[k];
                Stg &g = stg[slot_stg[k]];
                bool ok = !g.bad;
                for (int c = 0; ok && c < g.nct; c++) ok = lane->h_status[job[g.op0 + c]] != kJobFallback;
                if (!ok) {
                    redo[k] = 1;
                    return;
                }
                TileItem &it = items[i];
                if (pack_on_device && !h_cflag[k]) {
                    const uint8_t *frame = lane->h_outframes + k * kPackedFrameStride;
                    uint8_t *direct = nullptr;
                    if (it.take_malloc) {
                        it.out_malloc_len = wrapped_ciphertext_size(prep[i].va, kPackedFrameBytes);
                        direct = (uint8_t *)malloc(it.out_malloc_len);
                    }
                    if (direct) {
                        wrap_ciphertext_blob_to(prep[i].va, frame, kPackedFrameBytes, direct);
                        it.out_malloc = direct;
                    } else {
                        wrap_ciphertext_blob(prep[i].va, frame, kPackedFrameBytes, &it.out);
                    }
                    it.rc = kOk;
                } else if (!pack_on_device) {
                    it.rc = encode_ciphertext(prep[i].va, lane->h_out + k * kCtWords, &it.out);
                } else {
                    redo[k] = 2;  // constant result (a transparent ciphertext): the host writer's libzstd path, below
                }
                if (redo[k] == 0) prep[i].live = false;
            });
            for (size_t k = 0; k < slots; k++) {
                const size_t i = slot_item[k];
                if (redo[k] == 1) {
                    rest.push_back(i);
                } else if (redo[k] == 2) {
                    cuda_throw(cudaMemcpyAsync(lane->h_out + k * kCtWords, lane->d_out + k * kCtWords, kCtWords * 8, cudaMemcpyDeviceToHost, s),
                               "D2H");
                    cuda_throw(cudaStreamSynchronize(s), "stream sync");
                    items[i].rc = encode_ciphertext(prep[i].va, lane->h_out + k * kCtWords, &items[i].out);
                    prep[i].live = false;
                }
            }
        }
        std::stable_sort(rest.begin(), rest.end(), by_class);
        order.swap(rest);
    }

    // ---- host pass: operands into adjacent staging slots, class by class; a call that fails here gives its slot to the next
    std::vector<Run> runs;
    RunKeys run_keys;
    std::vector<size_t> slot_item;
    size_t slots = 0, ctct_slots = 0;
    for (size_t i : order) {
        TileItem &it = items[i];
        Prep &p = prep[i];
        uint64_t *ha = lane->h_a + slots * kCtWords;
        uint64_t *hb = lane->h_b + slots * kCtWords;
        uint16_t *hp = lane->h_plain + slots * kN;
        int32_t rc = 0;
        if (it.shape == Shape::CtCt) {
            CipherView vb;
            if (cnt == 1) {
                // a single call: inflate the second operand on a pool thread while this one inflates the first (a tile
                // already keeps every core busy).  If no pool thread is free the caller does both, in order.
                int32_t rcs[2] = {0, 0};
                std::atomic<int> next{0};
                const std::function<void()> fn = [&] {
                    for (int k; (k = next.fetch_add(1)) < 2;)
                        rcs[k] = k == 0 ? decode_ciphertext(p.sa, &p.va, ha) : decode_ciphertext(p.sb, &vb, hb);
                };
                HostPool::get().run(1, fn);
                rc = rcs[0] ? rcs[0] : rcs[1];  // reference order: a's error wins
            } else if (!(rc = decode_ciphertext(p.sa, &p.va, ha))) {
                rc = decode_ciphertext(p.sb, &vb, hb);
            }
            if (!rc && (!data_type_matches(p.va.data_type, it.kind) || !data_type_matches(vb.data_type, it.kind))) rc = kErrSunscreen;
        } else if (it.shape == Shape::CtPt) {
            if (!(rc = decode_ciphertext(p.sa, &p.va, ha)) && !(rc = encode_scalar(it.kind, p.sb, hp)))
                if (!data_type_matches(p.va.data_type, it.kind)) rc = kErrSunscreen;
        } else {
            if (!(rc = encode_scalar(it.kind, p.sa, hp)) && !(rc = decode_ciphertext(p.sb, &p.va, ha)))
                if (!data_type_matches(p.va.data_type, it.kind)) rc = kErrSunscreen;
        }
        if (!rc) rc = p.key_rc;
        if (rc) {
            it.rc = rc;
            p.live = false;
            continue;
        }
        if (p.cls == kMulCt) run_keys.add(p.d_rk);
        if (runs.empty() || runs.back().cls != p.cls) runs.push_back(Run{p.cls, slots, slots});
        runs.back().end = ++slots;
        if (p.cls <= kSubCt) ctct_slots = slots;
        slot_item.push_back(i);
    }
    if (slots == 0) return;
    const double t_decode = us_since(t_start);

    if (timed) cudaEventRecord(lane->ev[0], s);
    cuda_throw(cudaMemcpyAsync(lane->d_a, lane->h_a, slots * kCtWords * 8, cudaMemcpyHostToDevice, s), "H2D a");
    if (ctct_slots)
        cuda_throw(cudaMemcpyAsync(lane->d_b, lane->h_b, ctct_slots * kCtWords * 8, cudaMemcpyHostToDevice, s), "H2D b");
    if (slots > ctct_slots)
        cuda_throw(cudaMemcpyAsync(lane->d_plain + ctct_slots * kN, lane->h_plain + ctct_slots * kN, (slots - ctct_slots) * kN * 2,
                                   cudaMemcpyHostToDevice, s),
                   "H2D plain");
    if (timed) cudaEventRecord(lane->ev[1], s);
    launch_runs(runs, run_keys);
    if (timed) cudaEventRecord(lane->ev[2], s);
    cuda_throw(cudaMemcpyAsync(lane->h_out, lane->d_out, slots * kCtWords * 8, cudaMemcpyDeviceToHost, s), "D2H");
    if (timed) cudaEventRecord(lane->ev[3], s);
    cuda_throw(cudaStreamSynchronize(s), "stream sync");
    const double t_device = us_since(t_start);
    for (size_t k = 0; k < slots; k++) {
        TileItem &it = items[slot_item[k]];
        it.rc = encode_ciphertext(prep[slot_item[k]].va, lane->h_out + k * kCtWords, &it.out);
    }
    if (timed) {
        CallBreakdown &b = tl_breakdown;
        float ms[3] = {0, 0, 0};
        for (int k = 0; k < 3; k++) cudaEventElapsedTime(&ms[k], lane->ev[k], lane->ev[k + 1]);
        b.unpack_key_us = t_unpack;
        b.decode_us = t_decode - t_unpack;
        b.h2d_us = ms[0] * 1e3;
        b.kernels_us = ms[1] * 1e3;
        b.d2h_us = ms[2] * 1e3;
        b.total_us = us_since(t_start);
        b.encode_us = b.total_us - t_device;
    }
}

// ---------------------------------------------------------------- device-resident encrypt / decrypt
void Engine::encrypt_device(int device, const uint64_t *pk, const uint16_t *plain, const uint64_t *seeds, uint64_t *ct, size_t n,
                            cudaStream_t s) {
    encrypt_keyed_device(device, pk, nullptr, plain, seeds, ct, n, s);
}
void Engine::encrypt_keyed_device(int device, const uint64_t *pks, const int32_t *key_index, const uint16_t *plain,
                                  const uint64_t *seeds, uint64_t *ct, size_t n, cudaStream_t s) {
    device_context(device);
    if (n == 0) return;
    const size_t chunk = chunk_ops_ < n ? chunk_ops_ : n;
    ScratchLease lease{this, lease_scratch(device, s, chunk), &Engine::release_scratch};
    uint64_t *encbuf = lease.st->p;
    for (size_t off = 0; off < n; off += chunk) {
        const size_t c = n - off < chunk ? n - off : chunk;
        cuda_throw(launch_encrypt_keyed(pks, key_index ? key_index + off : nullptr, plain + off * kN, seeds + off * 8, encbuf,
                                        ct + off * kCtWords, c, s),
                   "encrypt");
    }
}
void Engine::decrypt_device(int device, const uint64_t *ct, const uint64_t *sk, uint16_t *plain, size_t n, cudaStream_t s,
                            int32_t *exhausted) {
    device_context(device);
    if (n == 0) return;
    const size_t chunk = chunk_ops_ < n ? chunk_ops_ : n;
    ScratchLease lease{this, lease_scratch(device, s, chunk), &Engine::release_scratch};
    uint64_t *xbuf = lease.st->p;
    for (size_t off = 0; off < n; off += chunk) {
        const size_t c = n - off < chunk ? n - off : chunk;
        cuda_throw(launch_decrypt(ct + off * kCtWords, sk, xbuf, plain + off * kN, c, s, exhausted ? exhausted + off : nullptr), "decrypt");
    }
}

// ---------------------------------------------------------------- threshold-network simulation API (fhe.rs:594-779)
namespace {
// the reference's private 512-bit constant mixed into the encrypt seed (fhe.rs:604-609)
const uint8_t kSeedConstant[64] = {15,  17,  225, 5,   30,  1,   237, 218, 130, 19,  37,  95,  222, 218, 244, 172,
                                   214, 175, 175, 110, 173, 103, 172, 60,  43,  76,  40,  150, 215, 96,  23,  78,
                                   22,  39,  30,  177, 107, 130, 124, 109, 27,  96,  206, 125, 104, 241, 10,  40,
                                   88,  238, 117, 118, 79,  113, 213, 110, 148, 179, 53,  19,  227, 154, 151, 122};
// the eight little-endian u64 words of SHA-512(msg) the reference hands to SEAL as the PRNG seed (fhe.rs:47-54, 611-616):
// all 512 bits reach the device sampler
struct Seed512 {
    uint64_t w[8];
};
Seed512 seed_from_hash(const std::vector<uint8_t> &msg) {
    uint8_t h[64];
    sha512(msg.data(), msg.size(), h);
    Seed512 s;
    memcpy(s.w, h, 64);
    return s;
}
}  // namespace

// encrypts the scalar operand `scalar` under `pk_bytes` with `seed`; uses the lane's plain / out buffers
int32_t Engine::encrypt_plain(Kind kind, Span scalar, Span pk_bytes, const uint64_t seed[8], CipherView *view, Lane *lane,
                              std::vector<uint8_t> *out) {
    int32_t rc = encode_scalar(kind, scalar, lane->h_plain);
    if (rc) return rc == kErrSunscreen ? kErrFailedEncryption : rc;
    const uint64_t *d_pk = nullptr;
    KeyPin pin;
    rc = public_key(pk_bytes, lane->device, &d_pk, &pin);
    if (rc) return rc;
    cudaStream_t s = lane->stream;
    memcpy(lane->h_b, seed, 64);
    cuda_throw(cudaMemcpyAsync(lane->d_plain, lane->h_plain, kN * 2, cudaMemcpyHostToDevice, s), "H2D plain");
    cuda_throw(cudaMemcpyAsync(lane->d_b, lane->h_b, 64, cudaMemcpyHostToDevice, s), "H2D seed");
    int *d_failed = reinterpret_cast<int *>(lane->d_scratch + 6 * kN);  // right behind the [6][N] encryption scratch
    cuda_throw(launch_encrypt(d_pk, lane->d_plain, lane->d_b, lane->d_scratch, lane->d_out, 1, s, d_failed), "encrypt");
    cuda_throw(cudaMemcpyAsync(lane->h_out, lane->d_out, kCtWords * 8, cudaMemcpyDeviceToHost, s), "D2H");
    cuda_throw(cudaMemcpyAsync(lane->h_b + 8, d_failed, sizeof(int), cudaMemcpyDeviceToHost, s), "D2H sampler flag");
    cuda_throw(cudaStreamSynchronize(s), "stream sync");
    if (*reinterpret_cast<const int *>(lane->h_b + 8)) return kErrFailedEncryption;  // PRNG stream window exhausted (~24 sigma)
    return encode_ciphertext(*view, lane->h_out, out);
}

int32_t Engine::encrypt(Kind kind, Span in, Span net_pub, Span, std::vector<uint8_t> *out) {
    Span plain, public_data;
    int32_t rc = unpack_two_arguments(in, &plain, &public_data);
    if (rc) return rc;
    // seed = SHA-512(public_data || constant || plain bytes)   (fhe.rs:600-611)
    std::vector<uint8_t> msg(public_data.p, public_data.p + public_data.n);
    msg.insert(msg.end(), kSeedConstant, kSeedConstant + 64);
    msg.insert(msg.end(), plain.p, plain.p + plain.n);
    Lane *lane = acquire_lane();
    LaneGuard guard{this, lane, &Engine::release_lane};
    cuda_throw(cudaSetDevice(lane->device), "cudaSetDevice");
    CipherView view;
    view.data_type = data_type_of(kind);
    testnet_params(view.params);
    return encrypt_plain(kind, plain, net_pub, seed_from_hash(msg).w, &view, lane, out);
}

int32_t Engine::decrypt(Kind kind, Span in, Span, Span net_pri, std::vector<uint8_t> *out) {
    Lane *lane = acquire_lane();
    LaneGuard guard{this, lane, &Engine::release_lane};
    cuda_throw(cudaSetDevice(lane->device), "cudaSetDevice");
    CipherView view;
    int32_t rc = decode_ciphertext(in, &view, lane->h_a);
    if (rc) return rc == kErrSunscreen ? kErrFailedDecryption : rc;
    if (!data_type_matches(view.data_type, kind)) return kErrFailedDecryption;  // fhe.rs:696 map_err
    const uint64_t *d_sk = network_sk(lane->device, net_pri);
    cudaStream_t s = lane->stream;
    cuda_throw(cudaMemcpyAsync(lane->d_a, lane->h_a, kCtWords * 8, cudaMemcpyHostToDevice, s), "H2D ct");
    int *d_flag = reinterpret_cast<int *>(lane->d_scratch + 2 * kN);  // right behind the [2][N] dot-product buffer
    cuda_throw(launch_decrypt(lane->d_a, d_sk, lane->d_scratch, lane->d_plain, 1, s, d_flag), "decrypt");
    cuda_throw(cudaMemcpyAsync(lane->h_plain, lane->d_plain, kN * 2, cudaMemcpyDeviceToHost, s), "D2H plain");
    cuda_throw(cudaMemcpyAsync(lane->h_out, d_flag, sizeof(int), cudaMemcpyDeviceToHost, s), "D2H noise flag");
    cuda_throw(cudaStreamSynchronize(s), "stream sync");
    // sunscreen's Runtime::decrypt refuses a ciphertext whose invariant noise budget is 0 (-> fhe.rs:643, 696)
    if (*reinterpret_cast<const int *>(lane->h_out)) return kErrFailedDecryption;
    decode_scalar(kind, lane->h_plain, kN, out);
    return kOk;
}

int32_t Engine::reencrypt(Kind kind, Span in, Span, Span net_pri, std::vector<uint8_t> *out) {
    Span pk, ct, public_data;
    int32_t rc = unpack_binary_operation(in, &pk, &ct, &public_data);
    if (rc) return rc;
    Lane *lane = acquire_lane();
    LaneGuard guard{this, lane, &Engine::release_lane};
    cuda_throw(cudaSetDevice(lane->device), "cudaSetDevice");
    // reference order: key, ciphertext, public data are all deserialised first (pack.rs:261-263)
    const uint64_t *d_pk = nullptr;
    KeyPin pin;  // validates the target key first, as the reference's unpack order does; encrypt_plain re-pins it
    if ((rc = public_key(pk, lane->device, &d_pk, &pin))) return rc;
    CipherView view;
    if ((rc = decode_ciphertext(ct, &view, lane->h_a))) return rc == kErrSunscreen ? kErrFailedDecryption : rc;
    if (!data_type_matches(view.data_type, kind)) return kErrFailedDecryption;
    const uint64_t *d_sk = network_sk(lane->device, net_pri);
    cudaStream_t s = lane->stream;
    cuda_throw(cudaMemcpyAsync(lane->d_a, lane->h_a, kCtWords * 8, cudaMemcpyHostToDevice, s), "H2D ct");
    int *d_flag = reinterpret_cast<int *>(lane->d_scratch + 2 * kN);  // right behind the [2][N] dot-product buffer
    cuda_throw(launch_decrypt(lane->d_a, d_sk, lane->d_scratch, lane->d_plain, 1, s, d_flag), "decrypt");
    cuda_throw(cudaMemcpyAsync(lane->h_plain, lane->d_plain, kN * 2, cudaMemcpyDeviceToHost, s), "D2H plain");
    cuda_throw(cudaMemcpyAsync(lane->h_out, d_flag, sizeof(int), cudaMemcpyDeviceToHost, s), "D2H noise flag");
    cuda_throw(cudaStreamSynchronize(s), "stream sync");
    // sunscreen's Runtime::decrypt refuses a ciphertext whose invariant noise budget is 0 (-> fhe.rs:643, 696)
    if (*reinterpret_cast<const int *>(lane->h_out)) return kErrFailedDecryption;
    std::vector<uint8_t> scalar;
    decode_scalar(kind, lane->h_plain, kN, &scalar);
    // seed = SHA-512(public_data || whole input || plain bytes)   (fhe.rs:676, 646-649)
    std::vector<uint8_t> msg(public_data.p, public_data.p + public_data.n);
    msg.insert(msg.end(), in.p, in.p + in.n);
    msg.insert(msg.end(), scalar.begin(), scalar.end());
    return encrypt_plain(kind, Span{scalar.data(), scalar.size()}, pk, seed_from_hash(msg).w, &view, lane, out);
}


// ---------------------------------------------------------------- threshold calls of the batch surface, a tile at a time
// (1) per call, on the host pool: framing, the target key of a reencrypt (pinned for the tile), the route of the ciphertext
// operand.  (2) one codec pass and one launch_decrypt over every decrypt / reencrypt operand.  (3) per call: the decrypted
// scalars, then the seeds and plaintexts of every encryption.  (4) one launch_encrypt_keyed over every encrypt / reencrypt row,
// each under its own key, and the result writer as binary_tile's.  A call whose operand is not a libzstd or structured frame of
// its kind, or that the device decoder hands back, is marked `single`: the caller runs it as the single call, which owns those
// codes, once the tile has released its lane.
void Engine::threshold_tile(ThresholdItem *items, size_t cnt, Span net_pub, Span net_pri) {
    for (size_t i = 0; i < cnt; i++) items[i].single = cnt == 1;  // a lone call gains nothing from the tile
    if (cnt < 2) return;
    Lane *lane = acquire_lane();
    LaneGuard guard{this, lane, &Engine::release_lane};
    threshold_on_lane(lane, items, cnt, net_pub, net_pri);
}

void Engine::threshold_on_lane(Lane *lane, ThresholdItem *items, size_t cnt, Span net_pub, Span net_pri) {
    cuda_throw(cudaSetDevice(lane->device), "cudaSetDevice");
    ensure_capacity(lane, cnt);
    ensure_codec(lane);
    cudaStream_t s = lane->stream;
    const size_t cap = lane->cap;
    struct Prep {
        Span a, b;             // encrypt: plain, public data; reencrypt: target key, public data
        Operand op;            // decrypt / reencrypt: the ciphertext
        const uint64_t *d_pk = nullptr;
        KeyPin pin;
        std::vector<uint8_t> scalar;  // reencrypt: the decrypted value
        bool live = false;
    };
    std::vector<Prep> prep(cnt);

    // (1)
    parallel_for(cnt, 4, [&](size_t i) {
        ThresholdItem &it = items[i];
        Prep &p = prep[i];
        it.rc = kOk;
        Span ct = it.in;
        if (it.op == Threshold::Encrypt) {
            p.live = (it.rc = unpack_two_arguments(it.in, &p.a, &p.b)) == kOk;
            return;
        }
        if (it.op == Threshold::Reencrypt) {  // reference order: key, ciphertext, public data (pack.rs:261-263)
            if ((it.rc = unpack_binary_operation(it.in, &p.a, &ct, &p.b))) return;
            if ((it.rc = public_key(p.a, lane->device, &p.d_pk, &p.pin))) return;
        }
        const Route r = classify_operand(ct, it.kind, &p.op);
        if (r == Route::Zstd || r == Route::Packed) p.live = true;
        else it.single = true;
    });

    // (2)
    std::vector<size_t> dec_item;
    std::vector<StageOperand> sop;
    for (size_t i = 0; i < cnt; i++)
        if (prep[i].live && items[i].op != Threshold::Encrypt) {
            sop.push_back(StageOperand{prep[i].op.route, prep[i].op.frame.n, (int32_t)dec_item.size(), 0});
            dec_item.push_back(i);
        }
    const size_t D = dec_item.size();
    if (D) {
        std::vector<int32_t> job(D);
        std::vector<uint8_t> bad(D, 0);
        const StagePlan plan = plan_codec_jobs(sop.data(), D, lane->h_jobs, job.data());
        parallel_for(D, 2, [&](size_t k) {
            if (!stage_operand(prep[dec_item[k]].op, lane->h_jobs, job[k], lane->h_frames, lane->h_payloads)) {
                bad[k] = 1;
                lane->h_jobs[job[k]].kind = kJobNone;
            }
        });
        if (plan.frame_bytes)
            cuda_throw(cudaMemcpyAsync(lane->d_frames, lane->h_frames, plan.frame_bytes, cudaMemcpyHostToDevice, s), "H2D frames");
        if (plan.payloads)
            cuda_throw(cudaMemcpyAsync(lane->d_payloads, lane->h_payloads, (size_t)plan.payloads * kPayloadStride, cudaMemcpyHostToDevice, s),
                       "H2D payloads");
        cuda_throw(cudaMemcpyAsync(lane->d_jobs, lane->h_jobs, (size_t)plan.jobs * sizeof(CodecJob), cudaMemcpyHostToDevice, s), "H2D jobs");
        cuda_throw(launch_codec_inflate(lane->d_frames, lane->d_payloads, lane->d_jobs, lane->d_status, lane->d_work, lane->d_prefix, lane->d_a,
                                        nullptr, plan.jobs, plan.any_zstd, plan.any_packed, plan.payloads > 0, s),
                   "codec inflate");
        int32_t *d_exh = lane->d_status + 2 * cap, *h_exh = lane->h_status + 2 * cap;  // behind the job status
        cuda_throw(launch_decrypt(lane->d_a, network_sk(lane->device, net_pri), lane->d_scratch, lane->d_plain, D, s, d_exh), "decrypt");
        uint16_t *h_dec = reinterpret_cast<uint16_t *>(lane->h_a);  // decrypted plaintexts; h_plain stages the encryptions' below
        cuda_throw(cudaMemcpyAsync(h_dec, lane->d_plain, D * kN * 2, cudaMemcpyDeviceToHost, s), "D2H plain");
        cuda_throw(cudaMemcpyAsync(h_exh, d_exh, D * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H noise flags");
        cuda_throw(cudaMemcpyAsync(lane->h_status, lane->d_status, (size_t)plan.jobs * sizeof(int32_t), cudaMemcpyDeviceToHost, s),
                   "D2H status");
        cuda_throw(cudaStreamSynchronize(s), "stream sync");
        // (3a) the decrypted scalars; a noise budget of 0 is sunscreen's decryption failure (fhe.rs:643, 696)
        parallel_for(D, 8, [&](size_t k) {
            const size_t i = dec_item[k];
            ThresholdItem &it = items[i];
            Prep &p = prep[i];
            p.live = false;
            if (bad[k] || lane->h_status[job[k]] == kJobFallback) it.single = true;
            else if (h_exh[k]) it.rc = kErrFailedDecryption;
            else if (it.op == Threshold::Decrypt) decode_scalar(it.kind, h_dec + k * kN, kN, &it.out);
            else decode_scalar(it.kind, h_dec + k * kN, kN, &p.scalar), p.live = true;
        });
    }

    // (3b) encryption rows: encrypts under the network key, reencrypts under their target keys
    std::vector<size_t> enc_item;
    std::vector<const uint64_t *> keys;  // distinct keys of the tile, in the order of their first row
    std::map<const uint64_t *, int32_t> key_slot;
    const uint64_t *d_net_pk = nullptr;
    KeyPin net_pin;
    uint64_t *h_seeds = lane->h_b;
    int32_t *h_kidx = reinterpret_cast<int32_t *>(lane->h_b + cap * 8);
    for (size_t i = 0; i < cnt; i++) {
        if (!prep[i].live) continue;
        const uint64_t *pk = prep[i].d_pk;
        if (items[i].op == Threshold::Encrypt) {
            if (!d_net_pk && public_key(net_pub, lane->device, &d_net_pk, &net_pin) != kOk)
                throw std::runtime_error("fhe_b200: embedded network public key is corrupt");
            pk = d_net_pk;
        }
        const auto ins = key_slot.emplace(pk, (int32_t)keys.size());
        if (ins.second) keys.push_back(pk);
        h_kidx[enc_item.size()] = ins.first->second;
        enc_item.push_back(i);
    }
    const size_t E = enc_item.size();
    if (E == 0) return;
    parallel_for(E, 4, [&](size_t e) {
        const size_t i = enc_item[e];
        ThresholdItem &it = items[i];
        Prep &p = prep[i];
        std::vector<uint8_t> msg(p.b.p, p.b.p + p.b.n);
        Span scalar = p.a;
        if (it.op == Threshold::Encrypt) {  // seed = SHA-512(public_data || constant || plain bytes)   (fhe.rs:600-611)
            msg.insert(msg.end(), kSeedConstant, kSeedConstant + 64);
            msg.insert(msg.end(), p.a.p, p.a.p + p.a.n);
        } else {  // seed = SHA-512(public_data || whole input || plain bytes)   (fhe.rs:676, 646-649)
            msg.insert(msg.end(), it.in.p, it.in.p + it.in.n);
            msg.insert(msg.end(), p.scalar.begin(), p.scalar.end());
            scalar = Span{p.scalar.data(), p.scalar.size()};
        }
        const int32_t rc = encode_scalar(it.kind, scalar, lane->h_plain + e * kN);
        if (rc) {  // the row still computes, on whatever its staging holds; nobody reads it
            it.rc = rc == kErrSunscreen ? kErrFailedEncryption : rc;
            p.live = false;
            return;
        }
        memcpy(h_seeds + e * 8, seed_from_hash(msg).w, 64);
    });

    // (4) per-lane layout inside d_scratch: sampler streams [cap][6][N] | seeds [cap][8] | key indices [cap] | keys [k][2][3][N].
    // The keys start on a 256-byte boundary whatever the lane's capacity: k_encrypt_seal reads them 16 bytes at a time.
    uint64_t *encbuf = lane->d_scratch, *d_seeds = encbuf + cap * 6 * kN;
    int32_t *d_kidx = reinterpret_cast<int32_t *>(d_seeds + cap * 8);
    uint64_t *d_keys = d_seeds + ((cap * 9 + 31) & ~(size_t)31);
    static_assert(6 * kN + 9 + 31 + 2 * 6 * kN <= kScratchLimbsPerOp * kN, "per call: its stream, seed, index, the padding and up to two keys (k <= cap + 1)");
    int32_t *d_failed = lane->d_status + cap, *h_failed = lane->h_status + cap;
    int32_t *d_cflag = lane->d_status + 2 * cap, *h_cflag = lane->h_status + 2 * cap;
    for (size_t j = 0; j < keys.size(); j++)
        cuda_throw(cudaMemcpyAsync(d_keys + j * kPkWords, keys[j], kPkWords * 8, cudaMemcpyDeviceToDevice, s), "D2D key");
    cuda_throw(cudaMemcpyAsync(lane->d_plain, lane->h_plain, E * kN * 2, cudaMemcpyHostToDevice, s), "H2D plain");
    cuda_throw(cudaMemcpyAsync(d_seeds, h_seeds, E * 64, cudaMemcpyHostToDevice, s), "H2D seeds");
    cuda_throw(cudaMemcpyAsync(d_kidx, h_kidx, E * sizeof(int32_t), cudaMemcpyHostToDevice, s), "H2D key indices");
    cuda_throw(launch_encrypt_keyed(d_keys, d_kidx, lane->d_plain, d_seeds, encbuf, lane->d_out, E, s, d_failed), "encrypt");
    const bool pack_on_device = zstd_writer() == 1;
    if (pack_on_device) {
        cuda_throw(launch_codec_pack(lane->d_out, lane->d_outframes, d_cflag, lane->d_prefix, (int)E, s), "codec pack");
        cuda_throw(cudaMemcpyAsync(lane->h_outframes, lane->d_outframes, E * kPackedFrameStride, cudaMemcpyDeviceToHost, s), "D2H frames");
        cuda_throw(cudaMemcpyAsync(h_cflag, d_cflag, E * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H flags");
    } else {
        cuda_throw(cudaMemcpyAsync(lane->h_out, lane->d_out, E * kCtWords * 8, cudaMemcpyDeviceToHost, s), "D2H");
    }
    cuda_throw(cudaMemcpyAsync(h_failed, d_failed, E * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H sampler flags");
    cuda_throw(cudaStreamSynchronize(s), "stream sync");
    const CipherView enc_view[4] = {result_view(Kind::U256), result_view(Kind::U64), result_view(Kind::I64), result_view(Kind::Frac64)};
    std::vector<uint8_t> constant(E, 0);
    parallel_for(E, 4, [&](size_t e) {
        const size_t i = enc_item[e];
        ThresholdItem &it = items[i];
        Prep &p = prep[i];
        if (!p.live) return;
        const CipherView &view = it.op == Threshold::Encrypt ? enc_view[(int)it.kind] : p.op.view;
        if (h_failed[e]) {
            it.rc = kErrFailedEncryption;  // PRNG stream window exhausted (~24 sigma)
        } else if (!pack_on_device) {
            it.rc = encode_ciphertext(view, lane->h_out + e * kCtWords, &it.out);
        } else if (h_cflag[e]) {
            constant[e] = 1;  // constant result (a transparent ciphertext): the host writer's libzstd path, below
        } else {
            const uint8_t *frame = lane->h_outframes + e * kPackedFrameStride;
            uint8_t *direct = nullptr;
            if (it.take_malloc) {
                it.out_malloc_len = wrapped_ciphertext_size(view, kPackedFrameBytes);
                direct = (uint8_t *)malloc(it.out_malloc_len);
            }
            if (direct) {
                wrap_ciphertext_blob_to(view, frame, kPackedFrameBytes, direct);
                it.out_malloc = direct;
            } else {
                wrap_ciphertext_blob(view, frame, kPackedFrameBytes, &it.out);
            }
            it.rc = kOk;
        }
    });
    for (size_t e = 0; e < E; e++)
        if (constant[e]) {
            const size_t i = enc_item[e];
            cuda_throw(cudaMemcpyAsync(lane->h_out, lane->d_out + e * kCtWords, kCtWords * 8, cudaMemcpyDeviceToHost, s), "D2H");
            cuda_throw(cudaStreamSynchronize(s), "stream sync");
            items[i].rc = encode_ciphertext(items[i].op == Threshold::Encrypt ? enc_view[(int)items[i].kind] : prep[i].op.view,
                                            lane->h_out, &items[i].out);
        }
}

}  // namespace fheb
