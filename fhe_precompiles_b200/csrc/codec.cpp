// See codec.h for the formats and their provenance.
#include "codec.h"

#include <dlfcn.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <stdexcept>

#include "context.h"

namespace fheb {

// ---------------------------------------------------------------- zstd via dlopen
namespace {
struct ZstdApi {
    void *handle = nullptr;
    size_t (*compressBound)(size_t) = nullptr;
    unsigned (*isError)(size_t) = nullptr;
    unsigned long long (*getFrameContentSize)(const void *, size_t) = nullptr;
    void *(*createCCtx)() = nullptr;
    size_t (*freeCCtx)(void *) = nullptr;
    size_t (*compressCCtx)(void *, void *, size_t, const void *, size_t, int) = nullptr;
    void *(*createDCtx)() = nullptr;
    size_t (*freeDCtx)(void *) = nullptr;
    size_t (*decompressDCtx)(void *, void *, size_t, const void *, size_t) = nullptr;
    bool ok = false;
};
ZstdApi g_z;
std::once_flag g_z_once;

void load_zstd() {
    const char *names[] = {"libzstd.so.1", "libzstd.so"};
    for (const char *n : names) {
        g_z.handle = dlopen(n, RTLD_NOW | RTLD_LOCAL);
        if (g_z.handle) break;
    }
    if (!g_z.handle) return;
#define LOAD(field, sym)                                           \
    g_z.field = (decltype(g_z.field))dlsym(g_z.handle, sym);       \
    if (!g_z.field) return;
    LOAD(compressBound, "ZSTD_compressBound");
    LOAD(isError, "ZSTD_isError");
    LOAD(getFrameContentSize, "ZSTD_getFrameContentSize");
    LOAD(createCCtx, "ZSTD_createCCtx");
    LOAD(freeCCtx, "ZSTD_freeCCtx");
    LOAD(compressCCtx, "ZSTD_compressCCtx");
    LOAD(createDCtx, "ZSTD_createDCtx");
    LOAD(freeDCtx, "ZSTD_freeDCtx");
    LOAD(decompressDCtx, "ZSTD_decompressDCtx");
#undef LOAD
    g_z.ok = true;
}
const ZstdApi &zapi() {
    std::call_once(g_z_once, load_zstd);
    return g_z;
}
struct ThreadCtx {
    void *c = nullptr, *d = nullptr;
    ~ThreadCtx() {
        if (c) g_z.freeCCtx(c);
        if (d) g_z.freeDCtx(d);
    }
};
thread_local ThreadCtx tl_ctx;

constexpr int kZstdLevel = 3;       // SEAL_DEFAULT compression level for zstd (ZSTD_CLEVEL_DEFAULT)
constexpr uint16_t kSealMagic = 0xA15E;
constexpr size_t kSealHeader = 16;
constexpr size_t kMaxInflate = 1u << 24;  // refuse absurd frames (largest legitimate blob is ~400 KB)

// ---- little-endian reader
struct Rd {
    const uint8_t *p;
    size_t n, pos = 0;
    bool fail = false;
    Rd(const uint8_t *p_, size_t n_) : p(p_), n(n_) {}
    bool need(size_t k) {
        if (fail || k > n - pos) {
            fail = true;
            return false;
        }
        return true;
    }
    uint8_t u8() {
        if (!need(1)) return 0;
        return p[pos++];
    }
    uint32_t u32() {
        if (!need(4)) return 0;
        uint32_t v;
        memcpy(&v, p + pos, 4);
        pos += 4;
        return v;
    }
    uint64_t u64v() {
        if (!need(8)) return 0;
        uint64_t v;
        memcpy(&v, p + pos, 8);
        pos += 8;
        return v;
    }
    const uint8_t *take(size_t k) {
        if (!need(k)) return nullptr;
        const uint8_t *r = p + pos;
        pos += k;
        return r;
    }
    bool done() const { return !fail && pos == n; }
};

void put_u64(std::vector<uint8_t> &o, uint64_t v) {
    uint8_t b[8];
    memcpy(b, &v, 8);
    o.insert(o.end(), b, b + 8);
}
void put_u32(std::vector<uint8_t> &o, uint32_t v) {
    uint8_t b[4];
    memcpy(b, &v, 4);
    o.insert(o.end(), b, b + 4);
}

struct SealHeader {
    uint8_t compr;
    uint64_t size;
};
bool parse_seal_header(const uint8_t *p, size_t n, SealHeader *h) {
    if (n < kSealHeader) return false;
    uint16_t magic;
    memcpy(&magic, p, 2);
    if (magic != kSealMagic || p[2] != kSealHeader) return false;
    if (p[3] != 4) return false;  // version_major (SEAL 4.x); minor p[4] not constrained
    h->compr = p[5];
    if (p[6] || p[7]) return false;
    memcpy(&h->size, p + 8, 8);
    return true;
}
void write_seal_header(uint8_t *p, uint8_t compr, uint64_t size) {
    uint16_t magic = kSealMagic;
    memcpy(p, &magic, 2);
    p[2] = (uint8_t)kSealHeader;
    p[3] = 4;
    p[4] = 0;
    p[5] = compr;
    p[6] = p[7] = 0;
    memcpy(p + 8, &size, 8);
}

// ---------------------------------------------------------------- structure-aware zstd frames for ciphertext payloads
// A SEAL ciphertext payload is a 97-byte prefix followed by little-endian 64-bit words that are residues of 36-bit
// primes: bytes 5..7 of every word are zero.  libzstd at SEAL's default level spends ~0.5-1.5 ms per ciphertext
// finding that out (and ends at ~88.5 KB); the structure can be written down directly as a standard zstd frame
// (RFC 8878) at memcpy speed and 82 KB:
//   block A : raw literals = prefix + word 0 + low 5 bytes of word 1, one sequence (LL 110, ML 3, offset 8) -- this
//             makes 8 the first repeat offset
//   block(s): raw literals = the low 5 bytes of every remaining word, one sequence per word (LL 5, ML 3, repeat
//             offset 1); all three symbol tables in RLE mode, so the sequence bitstream is the end marker alone.
// Any zstd decoder reads it (the reference's SEAL uses ZSTD_decompressStream); words >= 2^40 fall back to libzstd.
// The reader recognises exactly this layout and unpacks it directly; everything else goes to libzstd.
std::atomic<int> g_zstd_writer{-1};  // -1 unset (read FHE_B200_ZSTD_WRITER), 0 libzstd level 3 (default: SEAL's bytes), 1 structured frames
constexpr size_t kPackPrefix = kCtHeaderBytes;
constexpr size_t kBlockAContent = kPackPrefix + 16;
constexpr size_t kBlockALits = kPackPrefix + 13;
static_assert(kBlockALits >= 64 && kBlockALits < 128, "block A literal length must use LL code 25");
constexpr size_t kPackBlockWords = 16384;  // 128 KiB of content, zstd's Block_Maximum_Size
constexpr uint64_t kMask40 = (1ull << 40) - 1;

struct PackLayout {  // header bytes around the literal runs, shared by the writer and the recogniser
    static size_t frame_header(uint8_t *o, size_t content) {
        const uint8_t h[5] = {0x28, 0xB5, 0x2F, 0xFD, 0xA0};  // magic, single segment + 4-byte content size
        memcpy(o, h, 5);
        const uint32_t fcs = (uint32_t)content;
        memcpy(o + 5, &fcs, 4);
        return 9;
    }
    static size_t literals_header(uint8_t *o, size_t n) {  // Raw_Literals_Block
        if (n < 32) {
            o[0] = (uint8_t)(n << 3);
            return 1;
        }
        if (n < 4096) {
            const uint16_t v = (uint16_t)((1u << 2) | (n << 4));
            memcpy(o, &v, 2);
            return 2;
        }
        const uint32_t v = (uint32_t)((3u << 2) | (n << 4));
        memcpy(o, &v, 3);
        return 3;
    }
    static size_t seq_count(uint8_t *o, size_t n) {
        if (n < 128) {
            o[0] = (uint8_t)n;
            return 1;
        }
        if (n < 0x7F00) {
            o[0] = (uint8_t)((n >> 8) + 0x80);
            o[1] = (uint8_t)n;
            return 2;
        }
        o[0] = 0xFF;
        const uint16_t v = (uint16_t)(n - 0x7F00);
        memcpy(o + 1, &v, 2);
        return 3;
    }
    static void block_header(uint8_t *o, size_t size, bool last) {
        const uint32_t v = (uint32_t)((last ? 1u : 0u) | (2u << 1) | (size << 3));  // Compressed_Block
        memcpy(o, &v, 3);
    }
    // sequence section of block A: 1 sequence, RLE tables LL code 25 / OF code 3 / ML code 0; bitstream (read from the
    // top): offset extra 3 bits = 11 - 8, literal-length extra 6 bits = 110 - 64, under the end marker
    static size_t block_a_sequences(uint8_t *o) {
        const uint32_t bits = (uint32_t)(kBlockALits - 64) | (3u << 6) | (1u << 9);
        const uint8_t s[7] = {0x01, 0x54, 25, 3, 0, (uint8_t)bits, (uint8_t)(bits >> 8)};
        memcpy(o, s, 7);
        return 7;
    }
    // sequence section of a word block: m sequences, RLE tables LL code 5 / OF code 0 (repeat offset 1) / ML code 0
    static size_t word_sequences(uint8_t *o, size_t m) {
        size_t k = seq_count(o, m);
        const uint8_t s[5] = {0x54, 5, 0, 0, 0x01};
        memcpy(o + k, s, 5);
        return k + 5;
    }
};

// payload (prefix + 8*w bytes) -> zstd frame at dst (capacity >= len + 64).  0 when the payload does not have the shape.
size_t zstd_pack40(const uint8_t *src, size_t len, uint8_t *dst) {
    if (len < kBlockAContent || ((len - kPackPrefix) & 7) || len > 0xFFFFFFFFull) return 0;
    const size_t w = (len - kPackPrefix) / 8;
    if (w >= 16) {  // constant data (a transparent all-zero ciphertext) compresses to a few hundred bytes with libzstd
        uint64_t first, v, diff = 0;
        memcpy(&first, src + kPackPrefix, 8);
        for (size_t i = 1; i < 16; i++) {
            memcpy(&v, src + kPackPrefix + 8 * i, 8);
            diff |= v ^ first;
        }
        if (!diff) return 0;
    }
    uint64_t acc = 0;
    uint8_t *o = dst;
    o += PackLayout::frame_header(o, len);
    {  // block A
        uint8_t *bh = o;
        o += 3;
        o += PackLayout::literals_header(o, kBlockALits);
        memcpy(o, src, kBlockALits);
        o += kBlockALits;
        uint64_t w0, w1;
        memcpy(&w0, src + kPackPrefix, 8);
        memcpy(&w1, src + kPackPrefix + 8, 8);
        acc |= w0 | w1;
        o += PackLayout::block_a_sequences(o);
        PackLayout::block_header(bh, (size_t)(o - bh - 3), w == 2);
    }
    const uint8_t *in = src + kBlockAContent;
    for (size_t done = 2; done < w;) {
        const size_t m = std::min(kPackBlockWords, w - done);
        uint8_t *bh = o;
        o += 3;
        o += PackLayout::literals_header(o, 5 * m);
        for (size_t i = 0; i < m; i++) {  // 8-byte store, 5-byte stride: the 3 spill bytes are overwritten next
            uint64_t v;
            memcpy(&v, in + 8 * i, 8);
            acc |= v;
            memcpy(o + 5 * i, &v, 8);
        }
        o += 5 * m;
        in += 8 * m;
        done += m;
        o += PackLayout::word_sequences(o, m);
        PackLayout::block_header(bh, (size_t)(o - bh - 3), done == w);
    }
    if (acc & ~kMask40) return 0;
    return (size_t)(o - dst);
}

// the inverse, for frames with exactly that layout.  false: not ours (the caller hands the frame to libzstd)
bool zstd_unpack40(const uint8_t *src, size_t slen, std::vector<uint8_t> *out) {
    uint8_t hdr[16];
    if (slen < 9 + 3 + 2 + kBlockALits + 7) return false;
    uint32_t fcs;
    memcpy(&fcs, src + 5, 4);
    const size_t len = fcs;
    if (len < kBlockAContent || ((len - kPackPrefix) & 7) || len > kMaxInflate) return false;
    PackLayout::frame_header(hdr, len);
    if (memcmp(src, hdr, 9) != 0) return false;
    const size_t w = (len - kPackPrefix) / 8;
    // walk the headers first (cheap), then unpack
    size_t pos = 9;
    {
        const size_t lh = PackLayout::literals_header(hdr + 3, kBlockALits);
        const size_t body = lh + kBlockALits + 7;
        PackLayout::block_header(hdr, body, w == 2);
        if (memcmp(src + pos, hdr, 3 + lh) != 0) return false;
        PackLayout::block_a_sequences(hdr);
        if (memcmp(src + pos + 3 + lh + kBlockALits, hdr, 7) != 0) return false;
        pos += 3 + body;
    }
    out->resize(len + 8);  // 8 bytes of slack for the word-wide stores below
    uint8_t *dst = out->data();
    {
        const uint8_t *lit = src + 9 + 3 + 2;
        memcpy(dst, lit, kBlockALits);
        memset(dst + kBlockALits, 0, 3);
        // the match copies bytes 5..7 of word 0: they must be zero for the result to be what the fast path assumes
        if (dst[kPackPrefix + 5] | dst[kPackPrefix + 6] | dst[kPackPrefix + 7]) return false;
    }
    uint8_t *o = dst + kBlockAContent;
    for (size_t done = 2; done < w;) {
        const size_t m = std::min(kPackBlockWords, w - done);
        const size_t lh = PackLayout::literals_header(hdr + 3, 5 * m);
        uint8_t sq[8];
        const size_t sl = PackLayout::word_sequences(sq, m);
        const size_t body = lh + 5 * m + sl;
        if (pos + 3 + body > slen) return false;
        PackLayout::block_header(hdr, body, done + m == w);
        if (memcmp(src + pos, hdr, 3 + lh) != 0) return false;
        const uint8_t *lit = src + pos + 3 + lh;
        if (memcmp(lit + 5 * m, sq, sl) != 0) return false;
        for (size_t i = 0; i < m; i++) {  // 8-byte load (the sequence section follows the literals, sl >= 6 > 3)
            uint64_t v;
            memcpy(&v, lit + 5 * i, 8);
            v &= kMask40;
            memcpy(o + 8 * i, &v, 8);
        }
        o += 8 * m;
        done += m;
        pos += 3 + body;
    }
    if (pos != slen) return false;
    out->resize(len);
    return true;
}

// header walk of zstd_unpack40 without touching the literals: is this frame in the structured layout for `len` content bytes?
bool zstd_is_pack40(const uint8_t *src, size_t slen, size_t len) {
    uint8_t hdr[16];
    if (slen < 9 + 3 + 2 + kBlockALits + 7 || len < kBlockAContent || ((len - kPackPrefix) & 7)) return false;
    PackLayout::frame_header(hdr, len);
    if (memcmp(src, hdr, 9) != 0) return false;
    const size_t w = (len - kPackPrefix) / 8;
    size_t pos = 9;
    {
        const size_t lh = PackLayout::literals_header(hdr + 3, kBlockALits);
        const size_t body = lh + kBlockALits + 7;
        PackLayout::block_header(hdr, body, w == 2);
        if (memcmp(src + pos, hdr, 3 + lh) != 0) return false;
        PackLayout::block_a_sequences(hdr);
        if (memcmp(src + pos + 3 + lh + kBlockALits, hdr, 7) != 0) return false;
        const uint8_t *w0 = src + pos + 3 + lh + kPackPrefix;
        if (w0[5] | w0[6] | w0[7]) return false;
        pos += 3 + body;
    }
    for (size_t done = 2; done < w;) {
        const size_t m = std::min(kPackBlockWords, w - done);
        const size_t lh = PackLayout::literals_header(hdr + 3, 5 * m);
        uint8_t sq[8];
        const size_t sl = PackLayout::word_sequences(sq, m);
        const size_t body = lh + 5 * m + sl;
        if (pos + 3 + body > slen) return false;
        PackLayout::block_header(hdr, body, done + m == w);
        if (memcmp(src + pos, hdr, 3 + lh) != 0) return false;
        if (memcmp(src + pos + 3 + lh + 5 * m, sq, sl) != 0) return false;
        done += m;
        pos += 3 + body;
    }
    return pos == slen;
}

int zstd_writer_mode() {
    int m = g_zstd_writer.load(std::memory_order_relaxed);
    if (m < 0) {
        const char *e = getenv("FHE_B200_ZSTD_WRITER");
        m = (e && (!strcmp(e, "structured") || !strcmp(e, "1"))) ? 1 : 0;
        g_zstd_writer.store(m, std::memory_order_relaxed);
    }
    return m;
}

// SEAL blob -> decompressed payload.  `expect` = exact payload size required (0: any up to kMaxInflate)
int32_t seal_inflate(const uint8_t *blob, size_t len, size_t expect, std::vector<uint8_t> *out, uint8_t *compr_out) {
    SealHeader h;
    if (!parse_seal_header(blob, len, &h)) return kErrInvalidEncoding;
    if (h.size < kSealHeader || h.size > len) return kErrInvalidEncoding;
    const uint8_t *body = blob + kSealHeader;
    const size_t blen = (size_t)h.size - kSealHeader;
    if (compr_out) *compr_out = h.compr;
    if (h.compr == 0) {
        if (expect && blen != expect) return kErrInvalidEncoding;
        out->assign(body, body + blen);
        return kOk;
    }
    if (h.compr == 2) {
        if (zstd_unpack40(body, blen, out)) {
            if (expect && out->size() != expect) return kErrInvalidEncoding;
            return kOk;
        }
        const ZstdApi &z = zapi();
        if (!z.ok) throw std::runtime_error("fhe_b200: libzstd.so.1 is required to read SEAL blobs");
        unsigned long long sz = z.getFrameContentSize(body, blen);
        if (sz > kMaxInflate) return kErrInvalidEncoding;  // also covers ZSTD_CONTENTSIZE_UNKNOWN / ERROR
        if (expect && sz != expect) return kErrInvalidEncoding;
        out->resize((size_t)sz);
        if (!tl_ctx.d) tl_ctx.d = z.createDCtx();
        size_t r = z.decompressDCtx(tl_ctx.d, out->data(), out->size(), body, blen);
        if (z.isError(r) || r != sz) return kErrInvalidEncoding;
        return kOk;
    }
    if (h.compr == 1) {
        size_t cap = expect ? expect : kMaxInflate;
        out->resize(cap);
        uLongf dl = (uLongf)cap;
        int r = uncompress(out->data(), &dl, body, (uLong)blen);
        if (r != Z_OK || (expect && dl != expect)) return kErrInvalidEncoding;
        out->resize(dl);
        return kOk;
    }
    return kErrInvalidEncoding;
}

void seal_deflate(const uint8_t *payload, size_t len, uint8_t compr, std::vector<uint8_t> *out) {
    size_t packed = 0;
    if (compr == 0) {
        out->resize(kSealHeader + len);
        memcpy(out->data() + kSealHeader, payload, len);
    } else if (compr == 1) {
        uLongf cap = compressBound((uLong)len);
        out->resize(kSealHeader + cap);
        if (compress2(out->data() + kSealHeader, &cap, payload, (uLong)len, Z_DEFAULT_COMPRESSION) != Z_OK)
            throw std::runtime_error("fhe_b200: zlib compress failed");
        out->resize(kSealHeader + cap);
    } else if (zstd_writer_mode() == 1 && (out->resize(kSealHeader + len + 64), true) &&
               (packed = zstd_pack40(payload, len, out->data() + kSealHeader)) != 0) {
        out->resize(kSealHeader + packed);
    } else {
        const ZstdApi &z = zapi();
        if (!z.ok) throw std::runtime_error("fhe_b200: libzstd.so.1 is required to write SEAL blobs");
        size_t cap = z.compressBound(len);
        out->resize(kSealHeader + cap);
        if (!tl_ctx.c) tl_ctx.c = z.createCCtx();
        size_t r = z.compressCCtx(tl_ctx.c, out->data() + kSealHeader, cap, payload, len, kZstdLevel);
        if (z.isError(r)) throw std::runtime_error("fhe_b200: zstd compress failed");
        out->resize(kSealHeader + r);
    }
    write_seal_header(out->data(), compr, out->size());
}

// Params that differ from the testnet set: SEAL-valid ones deserialize in the reference and fail later in
// Runtime::run (code 7); garbage fails inside deserialize (code 3).  `p` points at N, k, then k primes, t.
int32_t foreign_params_code(const uint8_t *p, uint64_t k) {
    uint64_t n, t;
    memcpy(&n, p, 8);
    if (n < 1024 || n > 32768 || (n & (n - 1)) || k < 1 || k > 16) return kErrInvalidEncoding;
    for (uint64_t i = 0; i < k; i++) {
        uint64_t q;
        memcpy(&q, p + 16 + 8 * i, 8);
        if (q < 2 || (q >> 60) || q % (2 * n) != 1 || !is_prime_u64(q)) return kErrInvalidEncoding;
    }
    memcpy(&t, p + 16 + 8 * k, 8);
    if (t < 2 || (t >> 60)) return kErrInvalidEncoding;
    return kErrSunscreen;
}

// sunscreen Params (bincode): N, k, q_i.., t, scheme u32, security u32.  Must equal the testnet set.
bool params_are_testnet(const uint8_t *p) {
    uint64_t w[6];
    memcpy(w, p, 48);
    uint32_t s[2];
    memcpy(s, p + 48, 8);
    // the security level is not checked by SEAL arithmetic; scheme must be BFV (0)
    return w[0] == (uint64_t)kN && w[1] == 3 && w[2] == kModulus[MQ0] && w[3] == kModulus[MQ1] && w[4] == kModulus[MP] &&
           w[5] == kT && s[0] == 0;
}

// parses the fixed 97-byte ciphertext / public-key payload prefix
struct CtMeta {
    uint64_t parms_id[4];
    uint8_t ntt;
    uint64_t size, n, k;
    double scale;
    uint64_t corr;
    uint64_t count;
};
bool parse_ct_meta(const uint8_t *p, size_t len, CtMeta *m) {
    if (len < kCtHeaderBytes) return false;
    memcpy(m->parms_id, p, 32);
    m->ntt = p[32];
    memcpy(&m->size, p + 33, 8);
    memcpy(&m->n, p + 41, 8);
    memcpy(&m->k, p + 49, 8);
    memcpy(&m->scale, p + 57, 8);
    memcpy(&m->corr, p + 65, 8);
    SealHeader h;
    if (!parse_seal_header(p + 73, len - 73, &h) || h.compr != 0) return false;
    memcpy(&m->count, p + 89, 8);
    if (h.size != 24 + 8 * m->count) return false;
    return true;
}
}  // namespace

bool zstd_available() { return zapi().ok; }
void set_zstd_writer(int mode) { g_zstd_writer.store(mode ? 1 : 0, std::memory_order_relaxed); }
int zstd_writer() { return zstd_writer_mode(); }

// ---------------------------------------------------------------- framing
static uint32_t be32(const uint8_t *p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }

int32_t unpack_binary_operation(Span in, Span *pk, Span *a, Span *b) {
    if (in.n < 8) return kErrUnexpectedEOF;
    size_t ix1 = be32(in.p), ix2 = be32(in.p + 4);
    if (ix1 < 8 || ix2 < ix1 || ix2 > in.n) return kErrUnexpectedEOF;  // reference: slice panic
    *pk = Span{in.p + 8, ix1 - 8};
    *a = Span{in.p + ix1, ix2 - ix1};
    *b = Span{in.p + ix2, in.n - ix2};
    return kOk;
}
int32_t unpack_two_arguments(Span in, Span *a, Span *b) {
    if (in.n < 4) return kErrUnexpectedEOF;
    size_t ix1 = be32(in.p);
    if (ix1 < 4 || ix1 > in.n) return kErrUnexpectedEOF;
    *a = Span{in.p + 4, ix1 - 4};
    *b = Span{in.p + ix1, in.n - ix1};
    return kOk;
}

// ---------------------------------------------------------------- Ciphertext
int32_t parse_ciphertext_framing(Span in, CipherView *view, Span *blob_out) {
    Rd r(in.p, in.n);
    uint64_t slen = r.u64v();
    if (r.fail || slen > 4096) return kErrInvalidEncoding;
    const uint8_t *s = r.take((size_t)slen);
    if (!s) return kErrInvalidEncoding;
    view->data_type.assign((const char *)s, (size_t)slen);
    uint32_t variant = r.u32();
    uint64_t count = r.u64v();
    if (r.fail || variant != 0) return kErrInvalidEncoding;
    if (count != 1) return r.fail ? kErrInvalidEncoding : kErrSunscreen;  // all four types use one SEAL ciphertext
    const uint8_t *params = r.take(16);
    if (!params) return kErrInvalidEncoding;
    uint64_t k;
    memcpy(&k, params + 8, 8);
    if (k > 64 || !r.take((size_t)k * 8 + 16)) return kErrInvalidEncoding;
    uint64_t blen = r.u64v();
    const uint8_t *blob = r.take((size_t)blen);
    if (!blob || !r.done()) return kErrInvalidEncoding;
    if (k != 3 || !params_are_testnet(params)) return foreign_params_code(params, k);
    memcpy(view->params, params, kParamsBytes);
    *blob_out = Span{blob, (size_t)blen};
    return kOk;
}

int classify_ciphertext_blob(Span blob, Span *frame, uint8_t *compr) {
    SealHeader h;
    if (!parse_seal_header(blob.p, blob.n, &h) || h.size < kSealHeader || h.size > blob.n) return -1;
    *compr = h.compr;
    if (h.compr != 2) return 0;
    *frame = Span{blob.p + kSealHeader, (size_t)h.size - kSealHeader};
    return zstd_is_pack40(frame->p, frame->n, kCtHeaderBytes + 8 * kCtWords) ? 2 : 1;
}

bool inflate_ct_payload(Span frame, uint8_t *dst) {
    const ZstdApi &z = zapi();
    if (!z.ok) throw std::runtime_error("fhe_b200: libzstd.so.1 is required to read SEAL blobs");
    const size_t want = kCtHeaderBytes + 8 * kCtWords;
    if (z.getFrameContentSize(frame.p, frame.n) != want) return false;
    if (!tl_ctx.d) tl_ctx.d = z.createDCtx();
    const size_t r = z.decompressDCtx(tl_ctx.d, dst, want, frame.p, frame.n);
    return !z.isError(r) && r == want;
}

bool inflate_ct_blob(Span blob, uint8_t *dst) {
    SealHeader h;
    if (!parse_seal_header(blob.p, blob.n, &h) || h.size < kSealHeader || h.size > blob.n) return false;
    const Span body{blob.p + kSealHeader, (size_t)h.size - kSealHeader};
    const size_t want = kCtHeaderBytes + 8 * kCtWords;
    if (h.compr == 0) {
        if (body.n != want) return false;
        memcpy(dst, body.p, want);
        return true;
    }
    if (h.compr == 1) {
        uLongf dl = (uLongf)want;
        return uncompress(dst, &dl, body.p, (uLong)body.n) == Z_OK && dl == want;
    }
    return h.compr == 2 && inflate_ct_payload(body, dst);
}

void canonical_ct_prefix(uint8_t *p) {
    const HostContext &H = HostContext::get();
    memcpy(p, H.parms_id_data, 32);
    p[32] = 0;
    const uint64_t size = 2, n = kN, k = 2, corr = 1, count = kCtWords;
    const double scale = 1.0;
    memcpy(p + 33, &size, 8);
    memcpy(p + 41, &n, 8);
    memcpy(p + 49, &k, 8);
    memcpy(p + 57, &scale, 8);
    memcpy(p + 65, &corr, 8);
    write_seal_header(p + 73, 0, 24 + 8 * count);
    memcpy(p + 89, &count, 8);
}

size_t wrapped_ciphertext_size(const CipherView &view, size_t body_len) {
    return 8 + view.data_type.size() + 12 + kParamsBytes + 8 + kSealHeader + body_len;
}
void wrap_ciphertext_blob(const CipherView &view, const uint8_t *body, size_t body_len, std::vector<uint8_t> *out) {
    out->resize(wrapped_ciphertext_size(view, body_len));
    wrap_ciphertext_blob_to(view, body, body_len, out->data());
}
void wrap_ciphertext_blob_to(const CipherView &view, const uint8_t *body, size_t body_len, uint8_t *o) {
    const size_t blob = kSealHeader + body_len;
    const uint64_t dl = view.data_type.size(), one = 1, bl = blob;
    const uint32_t zero = 0;
    memcpy(o, &dl, 8), o += 8;
    memcpy(o, view.data_type.data(), dl), o += dl;
    memcpy(o, &zero, 4), o += 4;
    memcpy(o, &one, 8), o += 8;
    memcpy(o, view.params, kParamsBytes), o += kParamsBytes;
    memcpy(o, &bl, 8), o += 8;
    write_seal_header(o, view.compr_mode, blob);
    memcpy(o + kSealHeader, body, body_len);
}

int32_t decode_ciphertext(Span in, CipherView *view, uint64_t *words) {
    const HostContext &H = HostContext::get();
    Span blob_span;
    int32_t frc = parse_ciphertext_framing(in, view, &blob_span);
    if (frc) return frc;
    const uint8_t *blob = blob_span.p;
    const size_t blen = blob_span.n;

    thread_local std::vector<uint8_t> payload;
    int32_t rc = seal_inflate(blob, (size_t)blen, 0, &payload, &view->compr_mode);
    if (rc) return rc;
    CtMeta m;
    if (!parse_ct_meta(payload.data(), payload.size(), &m)) return kErrInvalidEncoding;
    // SEAL is_valid_for(): known parms_id at a data level, consistent sizes, BFV scale / correction factor
    if (memcmp(m.parms_id, H.parms_id_data, 32) != 0) return kErrInvalidEncoding;
    if (m.n != (uint64_t)kN || m.k != 2 || m.size < 2 || m.size > 16) return kErrInvalidEncoding;
    if (m.count != m.size * m.k * m.n || payload.size() != kCtHeaderBytes + 8 * m.count) return kErrInvalidEncoding;
    if (m.scale != 1.0 || m.corr != 1 || m.ntt > 1) return kErrInvalidEncoding;
    // shapes the precompile programs cannot run on -> SEAL/sunscreen runtime error
    if (m.size != 2 || m.ntt != 0) return kErrSunscreen;
    memcpy(words, payload.data() + kCtHeaderBytes, kCtWords * 8);
    for (int pl = 0; pl < 4; pl++) {
        const uint64_t q = kModulus[pl & 1];
        const uint64_t *w = words + (size_t)pl * kN;
        uint64_t bad = 0;
        for (int i = 0; i < kN; i++) bad |= (uint64_t)(w[i] >= q);
        if (bad) return kErrInvalidEncoding;
    }
    return kOk;
}

int32_t encode_ciphertext(const CipherView &view, const uint64_t *words, std::vector<uint8_t> *out) {
    thread_local std::vector<uint8_t> payload, blob;
    payload.resize(kCtHeaderBytes + kCtWords * 8);
    uint8_t *p = payload.data();
    canonical_ct_prefix(p);
    memcpy(p + kCtHeaderBytes, words, kCtWords * 8);
    seal_deflate(payload.data(), payload.size(), view.compr_mode, &blob);

    out->clear();
    out->reserve(8 + view.data_type.size() + 12 + kParamsBytes + 8 + blob.size());
    put_u64(*out, view.data_type.size());
    out->insert(out->end(), view.data_type.begin(), view.data_type.end());
    put_u32(*out, 0);
    put_u64(*out, 1);
    out->insert(out->end(), view.params, view.params + kParamsBytes);
    put_u64(*out, blob.size());
    out->insert(out->end(), blob.begin(), blob.end());
    return kOk;
}

// ---------------------------------------------------------------- keys
namespace {
// WithContext<T>: Params, u64 len, blob
bool read_with_context(Rd &r, const uint8_t **params, const uint8_t **blob, size_t *blen) {
    const uint8_t *head = r.take(16);
    if (!head) return false;
    uint64_t k;
    memcpy(&k, head + 8, 8);
    if (k > 64) return false;
    if (!r.take((size_t)k * 8 + 16)) return false;
    *params = head;
    uint64_t n = r.u64v();
    *blob = r.take((size_t)n);
    *blen = (size_t)n;
    return *blob != nullptr;
}
bool words_below(const uint8_t *src, size_t n_words, uint64_t q) {
    uint64_t bad = 0;
    for (size_t i = 0; i < n_words; i++) {
        uint64_t v;
        memcpy(&v, src + 8 * i, 8);
        bad |= (uint64_t)(v >= q);
    }
    return !bad;
}
// key-level size-2 NTT-form "ciphertext" payload (a SEAL PublicKey) -> [2][3][N]
bool decode_key_ct(const uint8_t *p, size_t len, const HostContext &H, uint64_t *dst) {
    CtMeta m;
    if (!parse_ct_meta(p, len, &m)) return false;
    if (memcmp(m.parms_id, H.parms_id_key, 32) != 0) return false;
    if (m.n != (uint64_t)kN || m.k != 3 || m.size != 2 || m.ntt != 1) return false;
    if (m.count != kPkWords || len != kCtHeaderBytes + 8 * m.count) return false;
    const uint8_t *src = p + kCtHeaderBytes;
    for (int pl = 0; pl < 6; pl++)
        if (!words_below(src + (size_t)pl * kN * 8, kN, kModulus[pl % 3])) return false;
    if (dst) memcpy(dst, src, kPkWords * 8);
    return true;
}
}  // namespace

int32_t decode_public_key(Span in, uint64_t *pk_words, uint64_t *rk_words, bool *has_relin) {
    const HostContext &H = HostContext::get();
    Rd r(in.p, in.n);
    const uint8_t *params, *blob;
    size_t blen;
    if (!read_with_context(r, &params, &blob, &blen)) return kErrInvalidEncoding;
    {
        uint64_t k;
        memcpy(&k, params + 8, 8);
        if (k != 3 || !params_are_testnet(params)) return foreign_params_code(params, k);
    }
    std::vector<uint8_t> payload;
    int32_t rc = seal_inflate(blob, blen, 0, &payload, nullptr);
    if (rc) return rc;
    if (!decode_key_ct(payload.data(), payload.size(), H, pk_words)) return kErrInvalidEncoding;

    // Option<WithContext<GaloisKeys>>: parsed for framing only (never used by the precompiles)
    uint8_t tag = r.u8();
    if (r.fail || tag > 1) return kErrInvalidEncoding;
    if (tag == 1) {
        if (!read_with_context(r, &params, &blob, &blen)) return kErrInvalidEncoding;
        SealHeader h;
        if (!parse_seal_header(blob, blen, &h)) return kErrInvalidEncoding;
    }
    // Option<WithContext<RelinearizationKeys>>
    tag = r.u8();
    if (r.fail || tag > 1) return kErrInvalidEncoding;
    if (has_relin) *has_relin = (tag == 1);
    if (tag == 1) {
        if (!read_with_context(r, &params, &blob, &blen)) return kErrInvalidEncoding;
        uint64_t k;
        memcpy(&k, params + 8, 8);
        if (k != 3 || !params_are_testnet(params)) return foreign_params_code(params, k);
        rc = seal_inflate(blob, blen, 0, &payload, nullptr);
        if (rc) return rc;
        // KSwitchKeys payload: parms_id, dim1, then per row: dim2, { SEAL header(compr none) + PublicKey payload }
        Rd k2(payload.data(), payload.size());
        const uint8_t *pid = k2.take(32);
        uint64_t dim1 = k2.u64v();
        if (!pid || k2.fail || memcmp(pid, H.parms_id_key, 32) != 0) return kErrInvalidEncoding;
        if (dim1 < 1 || dim1 > 16) return kErrInvalidEncoding;
        for (uint64_t row = 0; row < dim1; row++) {
            uint64_t dim2 = k2.u64v();
            if (k2.fail || dim2 > 16) return kErrInvalidEncoding;
            if (row == 0 && dim2 != 2) return kErrInvalidEncoding;  // decomposition count = |q| = 2
            for (uint64_t j = 0; j < dim2; j++) {
                const uint8_t *hdr = k2.take(kSealHeader);
                SealHeader h;
                if (!hdr || !parse_seal_header(hdr, kSealHeader, &h) || h.compr != 0 || h.size < kSealHeader)
                    return kErrInvalidEncoding;
                const uint8_t *body = k2.take((size_t)h.size - kSealHeader);
                if (!body) return kErrInvalidEncoding;
                uint64_t *dst = (row == 0 && rk_words) ? rk_words + (size_t)j * kPkWords : nullptr;
                if (!decode_key_ct(body, (size_t)h.size - kSealHeader, H, dst)) return kErrInvalidEncoding;
            }
        }
        if (!k2.done()) return kErrInvalidEncoding;
    }
    if (!r.done()) return kErrInvalidEncoding;
    return kOk;
}

int32_t decode_private_key(Span in, uint64_t *sk_words) {
    const HostContext &H = HostContext::get();
    Rd r(in.p, in.n);
    const uint8_t *params, *blob;
    size_t blen;
    if (!read_with_context(r, &params, &blob, &blen) || !r.done()) return kErrInvalidEncoding;
    std::vector<uint8_t> payload;
    int32_t rc = seal_inflate(blob, blen, 0, &payload, nullptr);
    if (rc) return rc;
    // SecretKey payload = Plaintext::save_members: parms_id, coeff_count, scale, DynArray
    Rd p(payload.data(), payload.size());
    const uint8_t *pid = p.take(32);
    uint64_t cc = p.u64v();
    p.take(8);
    const uint8_t *hdr = p.take(kSealHeader);
    uint64_t count = p.u64v();
    if (p.fail || !pid || !hdr || memcmp(pid, H.parms_id_key, 32) != 0 || cc != 3 * (uint64_t)kN || count != cc)
        return kErrInvalidEncoding;
    const uint8_t *data = p.take((size_t)count * 8);
    if (!data || !p.done()) return kErrInvalidEncoding;
    memcpy(sk_words, data, (size_t)count * 8);
    return kOk;
}

// ---------------------------------------------------------------- scalar encoders (sunscreen types)
// sunscreen's runtime compares every argument's Type (name, version, is_encrypted) with the compiled program's signature and
// fails with an argument-mismatch error otherwise (-> code 7, fhe.rs:28).  `#[derive(TypeName)]` names a type
// module_path!() + "::" + identifier WITHOUT generic arguments and stamps the sunscreen crate version, so Unsigned<1>
// (Unsigned64) and Unsigned<4> (Unsigned256) carry the SAME name and the reference cannot tell them apart.  The Unsigned
// spelling and the version are pinned by the reference's SHA-512 known answers (fhe.rs:2101-2244: the hashed bytes contain
// the string); Signed and Fractional come from the same derive.
const char *data_type_of(Kind kind) {
    switch (kind) {
        case Kind::I64: return "sunscreen::types::bfv::signed::Signed,0.8.1,true";
        case Kind::U64:
        case Kind::U256: return "sunscreen::types::bfv::unsigned::Unsigned,0.8.1,true";
        default: return "sunscreen::types::bfv::fractional::Fractional,0.8.1,true";
    }
}
bool data_type_matches(const std::string &dt, Kind kind) { return dt == data_type_of(kind); }

static uint64_t be_u64(const uint8_t *p) {
    uint64_t v = 0;
    for (int i = 0; i < 8; i++) v = (v << 8) | p[i];
    return v;
}

int32_t encode_scalar(Kind kind, Span b, uint16_t *plain) {
    memset(plain, 0, kN * sizeof(uint16_t));
    switch (kind) {
        case Kind::U64: {
            if (b.n != 8) return kErrInvalidEncoding;
            uint64_t v = be_u64(b.p);
            for (int i = 0; i < 64; i++) plain[i] = (uint16_t)((v >> i) & 1);
            return kOk;
        }
        case Kind::U256: {
            if (b.n != 32) return kErrInvalidEncoding;
            for (int w = 0; w < 4; w++) {  // big-endian: word 0 of the byte string is the most significant
                uint64_t v = be_u64(b.p + 8 * (3 - w));
                for (int i = 0; i < 64; i++) plain[64 * w + i] = (uint16_t)((v >> i) & 1);
            }
            return kOk;
        }
        case Kind::I64: {
            if (b.n != 8) return kErrInvalidEncoding;
            int64_t v = (int64_t)be_u64(b.p);
            uint64_t mag = v < 0 ? (uint64_t)0 - (uint64_t)v : (uint64_t)v;
            for (int i = 0; i < 64; i++) {
                uint64_t bit = (mag >> i) & 1;
                plain[i] = (uint16_t)(v < 0 ? bit * (kT - bit) : bit);
            }
            return kOk;
        }
        case Kind::Frac64: {
            if (b.n != 8) return kErrInvalidEncoding;
            uint64_t bits = be_u64(b.p);
            double v;
            memcpy(&v, &bits, 8);
            if (std::isnan(v) || std::isinf(v)) return kErrSunscreen;
            if (v == 0.0 || std::fpclassify(v) == FP_SUBNORMAL) return kOk;
            uint64_t mant = (bits & 0xFFFFFFFFFFFFFull) | (1ull << 52);
            int64_t power = (int64_t)((bits >> 52) & 0x7ff) - 1023;
            uint64_t sign = bits >> 63;
            if (power + 1 > 64) return kErrSunscreen;
            for (int i = 0; i < 53; i++) {
                uint64_t bit = (mant >> i) & 1;
                int64_t bp = power - (53 - i - 1);
                size_t idx = bp >= 0 ? (size_t)bp : (size_t)((int64_t)kN + bp);
                uint64_t sg = bp >= 0 ? sign : (sign ^ 1);
                plain[idx] = (uint16_t)(sg == 0 ? bit : (bit ? kT - bit : 0));
            }
            return kOk;
        }
    }
    return kErrInvalidEncoding;
}

void decode_scalar(Kind kind, const uint16_t *plain, size_t len, std::vector<uint8_t> *out) {
    const uint64_t cutoff = (kT + 1) / 2;
    auto put_be64 = [&](uint64_t v) {
        for (int i = 7; i >= 0; i--) out->push_back((uint8_t)(v >> (8 * i)));
    };
    out->clear();
    if (kind == Kind::U64 || kind == Kind::I64) {
        size_t bits = len < 64 ? len : 64;
        uint64_t val = 0;
        for (size_t i = 0; i < bits; i++) {
            uint64_t c = plain[i];
            if (c < cutoff)
                val += ((uint64_t)1 << i) * c;
            else
                val -= ((uint64_t)1 << i) * (kT - c);
        }
        put_be64(val);
    } else if (kind == Kind::U256) {
        size_t bits = len < 256 ? len : 256;
        uint64_t acc[4] = {0, 0, 0, 0};
        for (size_t i = 0; i < bits; i++) {
            uint64_t c = plain[i];
            bool neg = c >= cutoff;
            uint64_t mag = neg ? kT - c : c;
            uint64_t term[4] = {0, 0, 0, 0};
            size_t w = i / 64, s = i % 64;
            term[w] = mag << s;
            if (s && w + 1 < 4) term[w + 1] = mag >> (64 - s);
            unsigned carry = 0;
            for (int k = 0; k < 4; k++) {
                unsigned __int128 sub = (unsigned __int128)term[k] + carry;
                if (!neg) {
                    unsigned __int128 rr = (unsigned __int128)acc[k] + sub;
                    acc[k] = (uint64_t)rr;
                    carry = (unsigned)(rr >> 64);
                } else {
                    carry = (unsigned __int128)acc[k] < sub;
                    acc[k] = (uint64_t)((unsigned __int128)acc[k] - sub);
                }
            }
        }
        for (int w = 3; w >= 0; w--) put_be64(acc[w]);
    } else {
        double val = 0.0;
        size_t n = len < (size_t)kN ? len : (size_t)kN;
        for (size_t i = 0; i < n; i++) {
            int64_t power = i < 64 ? (int64_t)i : (int64_t)i - (int64_t)kN;
            double sign = power >= 0 ? 1.0 : -1.0;
            uint64_t c = plain[i];
            if (c < cutoff)
                val += sign * (double)c * std::exp2((double)power);
            else
                val -= sign * (double)(kT - c) * std::exp2((double)power);
        }
        uint64_t bits;
        memcpy(&bits, &val, 8);
        put_be64(bits);
    }
}

}  // namespace fheb
