// extern "C" surface: include/fhe_precompiles_b200.h.  Part 1 mirrors /root/reference/src/c_fhe.rs:8-141.
#pragma GCC visibility push(default)
#include "../../include/fhe_precompiles_b200.h"
#pragma GCC visibility pop

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <deque>
#include <exception>
#include <functional>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "codec_kernels.h"
#include "engine.h"
#include "host_pool.h"
#include "kernels.h"
#include "value_kernels.h"

using namespace fheb;

namespace {
thread_local std::string tl_error;

void set_error(const char *what) {
    tl_error = what ? what : "unknown error";
    static bool verbose = getenv("FHE_B200_QUIET") == nullptr;
    if (verbose) fprintf(stderr, "[fhe_precompiles_b200] %s\n", tl_error.c_str());
}

// c_fhe.rs:34-54: success -> malloc'd copy; failure -> NULL / 0 / code
int32_t finish(int32_t rc, const std::vector<uint8_t> &res, uint8_t **output, int64_t *output_length) {
    if (rc == 0) {
        uint8_t *buf = (uint8_t *)malloc(res.size() ? res.size() : 1);
        if (!buf) rc = kErrSunscreen;
        else {
            memcpy(buf, res.data(), res.size());
            *output = buf;
            *output_length = (int64_t)res.size();
            return 0;
        }
    }
    *output = nullptr;
    *output_length = 0;
    return rc;
}

template <class F>
int32_t guarded(F &&f, uint8_t **output, int64_t *output_length) {
    std::vector<uint8_t> res;
    int32_t rc;
    try {
        rc = f(&res);
    } catch (const std::exception &e) {
        set_error(e.what());
        rc = kErrSunscreen;
    } catch (...) {
        set_error("unknown exception");
        rc = kErrSunscreen;
    }
    return finish(rc, res, output, output_length);
}

int32_t run_binary(Op op, Shape shape, Kind kind, const uint8_t *bytes, size_t len, uint8_t **output, int64_t *output_length) {
    return guarded([&](std::vector<uint8_t> *res) { return Engine::get().binary_op(op, shape, kind, Span{bytes, len}, res); },
                   output, output_length);
}

// network keys (fhe.rs:118-119 include_bytes!): linked into the library by keys_blob.S
extern "C" const uint8_t fhe_b200_network_pub[];
extern "C" const uint8_t fhe_b200_network_pub_end[];
extern "C" const uint8_t fhe_b200_network_pri[];
extern "C" const uint8_t fhe_b200_network_pri_end[];

struct OpDesc {
    const char *name;
    int32_t (*fn)(const uint8_t *, size_t, uint8_t **, int64_t *);
};
}  // namespace

extern "C" {

#define BIN(name, OP, SHAPE, KIND)                                                                                   \
    int32_t c_fhe_##name(const uint8_t *bytes, size_t bytes_length, uint8_t **output, int64_t *output_length) {      \
        return run_binary(Op::OP, Shape::SHAPE, Kind::KIND, bytes, bytes_length, output, output_length);             \
    }
#define BIN_TYPE(T, KIND)                        \
    BIN(add_cipher##T##_cipher##T, Add, CtCt, KIND) \
    BIN(add_cipher##T##_##T, Add, CtPt, KIND)       \
    BIN(add_##T##_cipher##T, Add, PtCt, KIND)       \
    BIN(sub_cipher##T##_cipher##T, Sub, CtCt, KIND) \
    BIN(sub_cipher##T##_##T, Sub, CtPt, KIND)       \
    BIN(sub_##T##_cipher##T, Sub, PtCt, KIND)       \
    BIN(mul_cipher##T##_cipher##T, Mul, CtCt, KIND) \
    BIN(mul_cipher##T##_##T, Mul, CtPt, KIND)       \
    BIN(mul_##T##_cipher##T, Mul, PtCt, KIND)
BIN_TYPE(u256, U256)
BIN_TYPE(u64, U64)
BIN_TYPE(i64, I64)
BIN_TYPE(frac64, Frac64)

#define THRESH(name, FN, KIND)                                                                                       \
    int32_t c_fhe_##name(const uint8_t *bytes, size_t bytes_length, uint8_t **output, int64_t *output_length) {      \
        return guarded(                                                                                              \
            [&](std::vector<uint8_t> *res) {                                                                        \
                return Engine::get().FN(Kind::KIND, Span{bytes, bytes_length},                                      \
                                        Span{fhe_b200_network_pub, (size_t)(fhe_b200_network_pub_end - fhe_b200_network_pub)}, \
                                        Span{fhe_b200_network_pri, (size_t)(fhe_b200_network_pri_end - fhe_b200_network_pri)}, \
                                        res);                                                                       \
            },                                                                                                       \
            output, output_length);                                                                                  \
    }
#define THRESH_TYPE(T, KIND)           \
    THRESH(encrypt_##T, encrypt, KIND) \
    THRESH(reencrypt_##T, reencrypt, KIND) \
    THRESH(decrypt_##T, decrypt, KIND)
THRESH_TYPE(u256, U256)
THRESH_TYPE(u64, U64)
THRESH_TYPE(i64, I64)
THRESH_TYPE(frac64, Frac64)

// fhe.rs:701-703
int32_t c_fhe_public_key_bytes(const uint8_t *, size_t, uint8_t **output, int64_t *output_length) {
    std::vector<uint8_t> res(fhe_b200_network_pub, fhe_b200_network_pub_end);
    return finish(0, res, output, output_length);
}

void fhe_free(const uint8_t *bytes) { free((void *)bytes); }

const char *fhe_error(int32_t code) {
    switch (code) {  // lib.rs:33-44
        case 1: return "Unexpected end of file";
        case 2: return "Platform architecture invalid";
        case 3: return "Invalid encoding";
        case 4: return "Overflow in FHE program";
        case 5: return "Invalid decryption";
        case 6: return "Invalid encryption";
        case 7: return "Base sunscreen error";
        default: return "Unknown error";
    }
}

// ------------------------------------------------------------------------------------------------ part 2
const char *fhe_b200_last_error(void) { return tl_error.c_str(); }

int32_t fhe_b200_device_count(void) { return device_count(); }

int32_t fhe_b200_init(int32_t device) {
    try {
        device_context(device);
        return 0;
    } catch (const std::exception &e) {
        set_error(e.what());
        return -1;
    }
}
uint64_t fhe_b200_launch_count(void) { return launch_count() + codec_launch_count(); }

#define OPD(name) {#name, c_fhe_##name}
#define OPD_TYPE(T)                                                                                              \
    OPD(add_cipher##T##_cipher##T), OPD(add_cipher##T##_##T), OPD(add_##T##_cipher##T), OPD(sub_cipher##T##_cipher##T), \
        OPD(sub_cipher##T##_##T), OPD(sub_##T##_cipher##T), OPD(mul_cipher##T##_cipher##T), OPD(mul_cipher##T##_##T),  \
        OPD(mul_##T##_cipher##T)
static const OpDesc kOps[] = {OPD_TYPE(u256),     OPD_TYPE(u64),        OPD_TYPE(i64),       OPD_TYPE(frac64),
                              OPD(encrypt_u256),  OPD(encrypt_u64),     OPD(encrypt_i64),    OPD(encrypt_frac64),
                              OPD(reencrypt_u256), OPD(reencrypt_u64),  OPD(reencrypt_i64),  OPD(reencrypt_frac64),
                              OPD(decrypt_u256),  OPD(decrypt_u64),     OPD(decrypt_i64),    OPD(decrypt_frac64),
                              OPD(public_key_bytes)};
static const int kNumOps = (int)(sizeof(kOps) / sizeof(kOps[0]));

int32_t fhe_b200_op_index(const char *name) {
    if (!name) return -1;
    for (int i = 0; i < kNumOps; i++)
        if (strcmp(kOps[i].name, name) == 0) return i;
    return -1;
}
const char *fhe_b200_op_name(int32_t index) { return (index >= 0 && index < kNumOps) ? kOps[index].name : nullptr; }

// ops 0..35 of kOps are the binary precompiles, laid out type-major: index = 9 * type + 3 * op + shape
static bool binary_desc(int32_t index, Op *op, Shape *shape, Kind *kind) {
    if (index < 0 || index >= 36) return false;
    static const Kind kinds[4] = {Kind::U256, Kind::U64, Kind::I64, Kind::Frac64};
    *kind = kinds[index / 9];
    *op = (Op)((index % 9) / 3);
    *shape = (Shape)(index % 3);
    return true;
}

static size_t env_or(const char *name, size_t dflt) {
    const char *e = getenv(name);
    return (e && atoll(e) > 0) ? (size_t)atoll(e) : dflt;
}

int64_t fhe_b200_batch(fhe_b200_call *calls, size_t n, int32_t host_threads) {
    if (!calls || n == 0) return 0;
    // Workers take TILES of consecutive calls: the binary precompiles of a tile share one lane, one H2D / D2H per operand
    // array and one batched kernel sequence per operation class (Engine::binary_tile), so launch and synchronisation cost
    // is paid per tile, not per call.  Two workers per core: while one waits on its lane another runs the codec.
    size_t nt = host_threads > 0 ? (size_t)host_threads : 2 * (size_t)std::thread::hardware_concurrency();
    if (nt == 0) nt = 1;
    if (const char *e = getenv("FHE_B200_BATCH_THREADS"))
        if (host_threads <= 0 && atoi(e) > 0) nt = (size_t)atoi(e);
    size_t tile = Engine::get().tile_ops_for(n);
    const size_t big = Engine::get().big_tile_ops_for(n);
    bool serial_loops = true;
    size_t budget = 0;  // big tiles: the batch's thread budget, divided among the tile workers for their per-call loops
    if (Engine::get().device_codec() && big > tile && n >= 2 * big) {
        // a large batch: few big tiles (each stages its calls on the whole host pool and launches thousands of operand frames
        // at once), a handful of them in flight so that one tile's host phases overlap another's device phases
        tile = big;
        budget = nt;
        // six tiles in flight keep one GPU and the host pool busy (8, 10, 12 measured no better); with several GPUs in one
        // process, one more per extra GPU
        nt = std::min<size_t>(nt, env_or("FHE_B200_BIG_TILE_WORKERS", std::max<size_t>(6, Engine::get().lane_device_count() + 2)));
        serial_loops = false;
    } else {
        while (tile > 1 && (n + tile - 1) / tile < nt) tile /= 2;  // keep every worker busy on small batches
    }
    const size_t tiles = (n + tile - 1) / tile;
    if (nt > tiles) nt = tiles;
    std::atomic<size_t> next{0};
    std::atomic<int64_t> failed{0};
    if (nt < std::max<size_t>(2, std::thread::hardware_concurrency() / 2)) serial_loops = false;  // few workers: let tiles use idle cores
    // a batch that may use every core lets each big tile spread its loops over the whole pool (measured: 96 k calls/s against
    // 53 k with six threads per tile - a tile's phases run one after the other, so each must be short); a batch with a smaller
    // budget (one of several ranks on the host) divides it among its tile workers
    const size_t loop_width =
        (budget && budget < std::thread::hardware_concurrency()) ? std::max<size_t>(1, (budget + nt - 1) / nt) : 0;
    auto worker = [&]() {
        std::vector<TileItem> items;
        std::vector<size_t> which;
        struct SerialLoops {
            bool on;
            explicit SerialLoops(bool v, size_t width) : on(v) {
                if (on) Engine::set_thread_serial_loops(true);
                Engine::set_thread_loop_width(width);
            }
            ~SerialLoops() {
                if (on) Engine::set_thread_serial_loops(false);
                Engine::set_thread_loop_width(0);
            }
        } serial_guard(serial_loops, loop_width);
        for (;;) {
            const size_t t = next.fetch_add(1);
            if (t >= tiles) break;
            const size_t lo = t * tile, hi = std::min(n, lo + tile);
            items.clear();
            which.clear();
            for (size_t i = lo; i < hi; i++) {
                fhe_b200_call &c = calls[i];
                Op op;
                Shape shape;
                Kind kind;
                if (binary_desc(c.op, &op, &shape, &kind)) {
                    items.push_back(TileItem{op, shape, kind, Span{c.bytes, c.bytes_length}, {}, 0});
                    items.back().take_malloc = true;
                    which.push_back(i);
                } else if (c.op < 0 || c.op >= kNumOps) {
                    c.status = kErrSunscreen;
                    c.output = nullptr;
                    c.output_length = 0;
                } else {
                    c.status = kOps[c.op].fn(c.bytes, c.bytes_length, &c.output, &c.output_length);
                }
            }
            if (!items.empty()) {
                try {
                    Engine::get().binary_tile(items.data(), items.size());
                } catch (const std::exception &e) {
                    set_error(e.what());
                    for (auto &it : items) it.rc = kErrSunscreen;
                } catch (...) {
                    set_error("unknown exception");
                    for (auto &it : items) it.rc = kErrSunscreen;
                }
                // results into caller-owned buffers (a malloc + an 82 KB copy per call): shared with the pool when this worker
                // runs a big tile, like the tile's own per-call loops
                const auto finish_one = [&](size_t k) {
                    fhe_b200_call &c = calls[which[k]];
                    if (items[k].out_malloc) {  // written in place by the tile: the caller frees it with fhe_free
                        if (items[k].rc == 0) {
                            c.status = 0, c.output = items[k].out_malloc, c.output_length = (int64_t)items[k].out_malloc_len;
                            items[k].out_malloc = nullptr;
                            return;
                        }
                        free(items[k].out_malloc);
                        items[k].out_malloc = nullptr;
                    }
                    c.status = finish(items[k].rc, items[k].out, &c.output, &c.output_length);
                    std::vector<uint8_t>().swap(items[k].out);
                };
                if (!serial_loops && items.size() >= 64) {
                    std::atomic<size_t> nextk{0};
                    const std::function<void()> body = [&] {
                        for (size_t k; (k = nextk.fetch_add(8)) < items.size();)
                            for (size_t j = k; j < std::min(items.size(), k + 8); j++) finish_one(j);
                    };
                    const size_t width = std::min<size_t>(loop_width ? loop_width : std::thread::hardware_concurrency(), items.size() / 8);
                    if (width < 2) body();
                    else HostPool::get().run(width - 1, body);
                } else {
                    for (size_t k = 0; k < items.size(); k++) finish_one(k);
                }
            }
            for (size_t i = lo; i < hi; i++)
                if (calls[i].status) failed.fetch_add(1);
        }
    };
    if (nt <= 1) worker();
    else HostPool::get().run(nt - 1, worker);
    return failed.load();
}

#define DEV_GUARD(body)                  \
    try {                                \
        body;                            \
        return 0;                        \
    } catch (const std::exception &e) {  \
        set_error(e.what());             \
        return -1;                       \
    }

int32_t fhe_b200_add(int32_t device, const uint64_t *a, const uint64_t *b, uint64_t *out, size_t n, void *stream) {
    DEV_GUARD(device_context(device); cuda_throw(launch_eltwise(a, b, out, n, 0, (cudaStream_t)stream), "add"));
}
int32_t fhe_b200_sub(int32_t device, const uint64_t *a, const uint64_t *b, uint64_t *out, size_t n, void *stream) {
    DEV_GUARD(device_context(device); cuda_throw(launch_eltwise(a, b, out, n, 1, (cudaStream_t)stream), "sub"));
}
int32_t fhe_b200_negate(int32_t device, const uint64_t *a, uint64_t *out, size_t n, void *stream) {
    DEV_GUARD(device_context(device); cuda_throw(launch_eltwise(a, a, out, n, 2, (cudaStream_t)stream), "negate"));
}
int32_t fhe_b200_plain_addsub(int32_t device, const uint64_t *ct, const uint16_t *plain, uint64_t *out, size_t n,
                              int32_t mode, void *stream) {
    DEV_GUARD(device_context(device);
              cuda_throw(launch_plain_addsub(ct, plain, out, n, mode, (cudaStream_t)stream), "plain_addsub"));
}
int32_t fhe_b200_multiply_plain(int32_t device, const uint64_t *ct, const uint16_t *plain, uint64_t *out, size_t n,
                                void *stream) {
    DEV_GUARD(device_context(device); cuda_throw(launch_mul_plain(ct, plain, out, n, (cudaStream_t)stream), "mul_plain"));
}
int32_t fhe_b200_multiply(int32_t device, const uint64_t *a, const uint64_t *b, uint64_t *out3, size_t n, void *stream) {
    DEV_GUARD(Engine::get().multiply(device, a, b, out3, n, (cudaStream_t)stream));
}
int32_t fhe_b200_relinearize(int32_t device, const uint64_t *c3, const uint64_t *rk, uint64_t *out, size_t n, void *stream) {
    DEV_GUARD(Engine::get().relinearize(device, c3, rk, out, n, (cudaStream_t)stream));
}
int32_t fhe_b200_mul_relin(int32_t device, const uint64_t *a, const uint64_t *b, const uint64_t *rk, uint64_t *out,
                           size_t n, void *stream) {
    DEV_GUARD(Engine::get().mul_relin(device, a, b, rk, out, n, (cudaStream_t)stream));
}
int32_t fhe_b200_int_peak(int32_t device, int32_t wide, double *tera_mads_per_s) {
    DEV_GUARD(device_context(device); cuda_throw(measure_int_peak(wide, tera_mads_per_s), "int_peak"));
}
int32_t fhe_b200_encrypt(int32_t device, const uint64_t *pk, const uint16_t *plain, const uint64_t *seeds, uint64_t *ct, size_t n,
                         void *stream) {
    DEV_GUARD(Engine::get().encrypt_device(device, pk, plain, seeds, ct, n, (cudaStream_t)stream));
}
int32_t fhe_b200_seal_sample(int32_t device, uint64_t *streams, int32_t *failed, size_t n, void *stream) {
    DEV_GUARD(device_context(device); cuda_throw(launch_seal_sample(streams, nullptr, failed, n, (cudaStream_t)stream), "seal_sample"));
}
size_t fhe_b200_seal_op_words(void) { return kSealOpWords; }
int32_t fhe_b200_decrypt(int32_t device, const uint64_t *ct, const uint64_t *sk, uint16_t *plain, size_t n, void *stream) {
    DEV_GUARD(Engine::get().decrypt_device(device, ct, sk, plain, n, (cudaStream_t)stream));
}
int32_t fhe_b200_decrypt_checked(int32_t device, const uint64_t *ct, const uint64_t *sk, uint16_t *plain, int32_t *exhausted, size_t n,
                                 void *stream) {
    DEV_GUARD(Engine::get().decrypt_device(device, ct, sk, plain, n, (cudaStream_t)stream, exhausted));
}
static void check_value_args(const char *fn, int32_t kind, const uint16_t *plain) {
    if (!value_kind_valid(kind))
        throw std::runtime_error(std::string(fn) + ": unknown kind " + std::to_string(kind) + " (0 u256, 1 u64, 2 i64, 3 frac64)");
    if ((uintptr_t)plain % 16) throw std::runtime_error(std::string(fn) + ": plain must be 16-byte aligned");
}
int32_t fhe_b200_encode_values(int32_t device, int32_t kind, const void *values, uint16_t *plain, int32_t *status, size_t n,
                               void *stream) {
    DEV_GUARD(check_value_args("fhe_b200_encode_values", kind, plain); device_context(device);
              cuda_throw(launch_encode_values(kind, values, plain, status, n, (cudaStream_t)stream), "encode_values"));
}
int32_t fhe_b200_decode_values(int32_t device, int32_t kind, const uint16_t *plain, void *values, size_t n, void *stream) {
    DEV_GUARD(check_value_args("fhe_b200_decode_values", kind, plain); device_context(device);
              cuda_throw(launch_decode_values(kind, plain, values, n, (cudaStream_t)stream), "decode_values"));
}
int32_t fhe_b200_bfly_peak(int32_t device, int32_t mod, double *giga_bfly_per_s) {
    DEV_GUARD(device_context(device); cuda_throw(measure_bfly_peak(mod, giga_bfly_per_s), "bfly_peak"));
}
int32_t fhe_b200_data_type_kind(const char *data_type) {
    if (!data_type) return -1;
    const std::string dt(data_type);
    for (int k = 0; k < 4; k++)
        if (data_type_matches(dt, (Kind)k)) return k;
    return -1;
}
int64_t fhe_b200_set_chunk_ops(int64_t ops) {
    try {
        return (int64_t)Engine::get().set_chunk_ops(ops);
    } catch (const std::exception &e) {
        set_error(e.what());
        return -1;
    }
}
void fhe_b200_set_call_timing(int32_t on) {
    try {
        Engine::get().set_call_timing(on != 0);
    } catch (...) {
    }
}
void fhe_b200_last_call_breakdown(double us[7]) {
    const CallBreakdown &b = Engine::last_call_breakdown();
    const double v[7] = {b.unpack_key_us, b.decode_us, b.h2d_us, b.kernels_us, b.d2h_us, b.encode_us, b.total_us};
    for (int i = 0; i < 7; i++) us[i] = v[i];
}
void fhe_b200_set_kernel_timing(int32_t on) {
    try {
        Engine::get().set_kernel_timing(on != 0);
    } catch (const std::exception &e) {
        set_error(e.what());
    }
}
int32_t fhe_b200_kernel_timing_report(int32_t device, double ms[16], uint64_t launches[16]) {
    DEV_GUARD(Engine::get().kernel_timing_report(device, ms, launches));
}
int32_t fhe_b200_mul_relin_host(int32_t device, const uint64_t *a, const uint64_t *b, const uint64_t *rk, uint64_t *out,
                                size_t n) {
    DEV_GUARD(Engine::get().mul_relin_host(device, a, b, rk, out, n));
}
int32_t fhe_b200_mul_relin_frames(int32_t device, const uint8_t *a_frames, const uint8_t *b_frames, size_t stride, const uint64_t *rk,
                                  uint8_t *out_frames, size_t n, int32_t *status) {
    DEV_GUARD(Engine::get().mul_relin_frames(device, a_frames, b_frames, stride, rk, out_frames, n, status));
}
int32_t fhe_b200_upload_frames(int32_t device, const uint8_t *frames, size_t stride, size_t n, uint64_t *d_words, int32_t *status) {
    DEV_GUARD(Engine::get().upload_frames(device, frames, stride, n, d_words, status));
}
int32_t fhe_b200_download_frames(int32_t device, const uint64_t *d_words, size_t n, uint8_t *out_frames, int32_t *status) {
    DEV_GUARD(Engine::get().download_frames(device, d_words, n, out_frames, status));
}
size_t fhe_b200_frame_bytes(void) { return kPackedFrameBytes; }
size_t fhe_b200_frame_stride(void) { return kPackedFrameStride; }
int32_t fhe_b200_ntt(int32_t device, uint64_t *data, size_t n_limbs, const int32_t *mods, int32_t n_mods, int32_t inverse,
                     void *stream) {
    if (!mods || n_mods < 1 || n_mods > kNumMod) {
        set_error("fhe_b200_ntt: n_mods must be 1..6");
        return -1;
    }
    LimbMods lm;
    lm.n = n_mods;
    for (int i = 0; i < kNumMod; i++) lm.mod[i] = 0;
    for (int i = 0; i < n_mods; i++) {
        if (mods[i] < 0 || mods[i] >= kNumMod) {
            set_error("fhe_b200_ntt: bad modulus index");
            return -1;
        }
        lm.mod[i] = mods[i];
    }
    DEV_GUARD(device_context(device); cuda_throw(launch_ntt(data, n_limbs, lm, inverse != 0, (cudaStream_t)stream), "ntt"));
}

int32_t fhe_b200_parse_public_key(const uint8_t *bytes, size_t len, uint64_t *pk_words, uint64_t *rk_words) {
    try {
        bool has = false;
        int32_t rc = decode_public_key(Span{bytes, len}, pk_words, rk_words, &has);
        if (rc == 0 && rk_words && !has) return kErrSunscreen;
        return rc;
    } catch (const std::exception &e) {
        set_error(e.what());
        return kErrSunscreen;
    }
}
int32_t fhe_b200_parse_private_key(const uint8_t *bytes, size_t len, uint64_t *sk_words) {
    try {
        return decode_private_key(Span{bytes, len}, sk_words);
    } catch (const std::exception &e) {
        set_error(e.what());
        return kErrSunscreen;
    }
}
int32_t fhe_b200_parse_ciphertext(const uint8_t *bytes, size_t len, uint64_t *words, char *data_type, size_t cap) {
    try {
        CipherView v;
        int32_t rc = decode_ciphertext(Span{bytes, len}, &v, words);
        if (rc == 0 && data_type && cap) {
            size_t k = v.data_type.size() < cap - 1 ? v.data_type.size() : cap - 1;
            memcpy(data_type, v.data_type.data(), k);
            data_type[k] = 0;
        }
        return rc;
    } catch (const std::exception &e) {
        set_error(e.what());
        return kErrSunscreen;
    }
}
int32_t fhe_b200_write_ciphertext(const uint64_t *words, const char *data_type, uint8_t **output, int64_t *output_length) {
    return guarded(
        [&](std::vector<uint8_t> *res) {
            CipherView v;
            v.data_type = data_type ? data_type : "";
            // testnet Params (testnet.rs:8-14) in sunscreen's bincode layout
            uint64_t w[6] = {(uint64_t)kN, 3, kModulus[MQ0], kModulus[MQ1], kModulus[MP], kT};
            memcpy(v.params, w, 48);
            memset(v.params + 48, 0, 8);
            v.compr_mode = 2;
            return encode_ciphertext(v, words, res);
        },
        output, output_length);
}
int32_t fhe_b200_zstd_inflate(int32_t device, const uint8_t *const *frames, const size_t *lens, size_t n, uint8_t *out,
                              int32_t *status, float *elapsed_ms) {
    try {
        device_context(device);
        std::vector<CodecJob> jobs(n);
        std::vector<uint8_t> staged(n * kFrameSlotBytes, 0);
        for (size_t i = 0; i < n; i++) {
            const bool fits = lens[i] + 2 * kFramePad <= kFrameSlotBytes;
            jobs[i] = CodecJob{i * kFrameSlotBytes + kFramePad, (uint32_t)(fits ? lens[i] : 0), fits ? kJobZstd : kJobNone, (int32_t)i, 0};
            if (fits) memcpy(staged.data() + jobs[i].src_off, frames[i], lens[i]);
        }
        uint8_t *d_frames = nullptr, *d_payloads = nullptr, *d_prefix = nullptr;
        CodecJob *d_jobs = nullptr;
        int32_t *d_status = nullptr;
        void *d_work = nullptr;
        cuda_throw(cudaMalloc((void **)&d_frames, staged.size()), "cudaMalloc");
        cuda_throw(cudaMalloc((void **)&d_payloads, n * kPayloadStride), "cudaMalloc");
        cuda_throw(cudaMalloc((void **)&d_jobs, n * sizeof(CodecJob)), "cudaMalloc");
        cuda_throw(cudaMalloc((void **)&d_status, n * 4), "cudaMalloc");
        cuda_throw(cudaMalloc(&d_work, n * codec_work_bytes()), "cudaMalloc");
        cuda_throw(cudaMalloc((void **)&d_prefix, kCtPrefixBytes), "cudaMalloc");
        cuda_throw(cudaMemset(d_status, 0, n * 4), "memset");
        cuda_throw(cudaMemset(d_prefix, 0, kCtPrefixBytes), "memset");
        cuda_throw(cudaMemcpy(d_frames, staged.data(), staged.size(), cudaMemcpyHostToDevice), "H2D");
        cuda_throw(cudaMemcpy(d_jobs, jobs.data(), n * sizeof(CodecJob), cudaMemcpyHostToDevice), "H2D");
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0), cudaEventCreate(&e1);
        for (int rep = 0; rep < 6; rep++) {  // the last repetition is timed: the first ones bring the clocks up
            cudaEventRecord(e0, nullptr);
            cuda_throw(launch_codec_inflate(d_frames, d_payloads, d_jobs, d_status, d_work, d_prefix, nullptr, nullptr, (int)n, true, false, false,
                                            nullptr),
                       "inflate");
            cudaEventRecord(e1, nullptr);
        }
        cuda_throw(cudaDeviceSynchronize(), "sync");
        if (elapsed_ms) cudaEventElapsedTime(elapsed_ms, e0, e1);
        cudaEventDestroy(e0), cudaEventDestroy(e1);
        cuda_throw(cudaMemcpy2D(out, kCtPayloadBytes, d_payloads, kPayloadStride, kCtPayloadBytes, n, cudaMemcpyDeviceToHost), "D2H");
        cuda_throw(cudaMemcpy(status, d_status, n * 4, cudaMemcpyDeviceToHost), "D2H");
        for (size_t i = 0; i < n; i++)
            if (status[i] != kJobOk) status[i] = kJobFallback;  // (frames too large to stage were never tried)
        cudaFree(d_frames), cudaFree(d_payloads), cudaFree(d_jobs), cudaFree(d_status), cudaFree(d_work), cudaFree(d_prefix);
        return 0;
    } catch (const std::exception &e) {
        set_error(e.what());
        return -1;
    }
}
void fhe_b200_sha512(const uint8_t *bytes, size_t len, int32_t portable, uint8_t out[64]) {
    if (portable) fheb::sha512_portable(bytes, len, out);
    else fheb::sha512(bytes, len, out);
}
int32_t fhe_b200_set_zstd_writer(int32_t mode) {
    int32_t prev = fheb::zstd_writer();
    if (mode >= 0) fheb::set_zstd_writer(mode);
    return prev;
}
void fhe_b200_parms_id(int32_t which, uint64_t out[4]) {
    try {
        const HostContext &H = HostContext::get();
        memcpy(out, which == 0 ? H.parms_id_key : H.parms_id_data, 32);
    } catch (...) {
        memset(out, 0, 32);
    }
}

}  // extern "C"
