// Shared parsing layer of the device zstd (RFC 8878) decoder: bit readers, FSE and Huffman table construction, and the
// literal-length / match-length codes.  zstd_plan2.h (parse, Huffman streams, sequences) and zstd_plan3.cuh / zstd_exec3.h
// (execution) build the decoder on it.  SURVEY 8f-3: the byte surface is bound by the host's libzstd inflate of the two
// ciphertext operands of every call; with this the compressed frames go over PCIe as they are and are inflated on the device,
// thousands at a time.  Aligned word loads only, all tables in a caller-provided workspace.
//
// Contract: anything the decoder does not reproduce EXACTLY as libzstd would -- dictionaries, checksums, several frames,
// unknown content size, offsets beyond the window, an over- or under-consumed bitstream, any malformed field -- is reported
// as kZdFallback and the caller hands that operand to libzstd on the host, whose verdict (payload or error code) is the
// one returned.  kZdOk therefore always means "byte-identical to libzstd's output".
//
// The same source compiles for the host (tests/test_zstd_dec.py drives it through tests/zd_host.cpp against libzstd on
// fixtures, random data at many levels and corrupted frames) and for the device (codec_kernels.cu).
// Buffers: `src` must be readable from kPad bytes before to kPad bytes after the frame (the bit readers use aligned
// word loads); the padding's content is irrelevant.
#pragma once
#include <cstddef>
#include <cstdint>

#if defined(__CUDACC__)
#define ZD_HD __host__ __device__ __forceinline__
#define ZD_FN __host__ __device__
#else
#define ZD_HD inline
#define ZD_FN inline
struct uint2 {  // host build: a sequence-table cell as the device loads it (zstd_plan2.h pack_cell)
    unsigned x, y;
};
#endif

namespace fheb {
namespace zd {

constexpr int kZdOk = 0;
constexpr int kZdFallback = 1;

constexpr size_t kBlockMax = 128 * 1024;
constexpr int kMaxLL = 35, kMaxML = 52, kMaxOF = 31;
constexpr int kHufLogMax = 11;
constexpr size_t kPad = 16;

struct FseEntry {  // plain FSE decoding cell (Huffman weights)
    uint8_t sym, nb;
    uint16_t base;
};
struct SeqEntry {  // sequence-table cell with the symbol already translated (like libzstd's ZSTD_seqSymbol)
    uint16_t next_base;   // next state = next_base + read(nb)
    uint8_t nb;
    uint8_t add_bits;     // extra bits of the value
    uint32_t base_value;  // literal length / match length base, or 1 << offset code
};

constexpr size_t kSeqTableEntries = 512 + 256 + 512;

struct Work {
    SeqEntry *ll, *of, *ml;  // where seq_table builds the three sequence tables: `store`, or a block's slot (zstd_plan2.h)
    SeqEntry store[kSeqTableEntries];
    FseEntry tmp[512];  // table under construction
    uint16_t huf[1 << kHufLogMax];  // sym | nb << 8
    int ll_log, of_log, ml_log, huf_log;
    int have_ll, have_of, have_ml, have_huf;
    // scratch for table construction
    int16_t norm[256];
    uint16_t state_desc[256];
    uint8_t weights[256];
    FseEntry wt[64];  // FSE table of the Huffman weights (accuracy log <= 6)
    uint8_t lit[kBlockMax + 8];
};

ZD_HD void work_bind(Work *w, SeqEntry *tables) {  // tables: kSeqTableEntries cells, or null to use w->store
    SeqEntry *t = tables ? tables : w->store;
    w->ll = t;
    w->of = t + 512;
    w->ml = t + 768;
}

// ---------------------------------------------------------------- bit access on aligned words
// 64 bits of the stream starting at bit `bit` (>= 0), little-endian bit order; `p` is the first byte of the stream
ZD_HD uint64_t window_at(const uint8_t *p, uint64_t bit) {
    const uintptr_t addr = (uintptr_t)p + (bit >> 3);
    const uint64_t *w = (const uint64_t *)(addr & ~(uintptr_t)7);
    const unsigned sh = (unsigned)((addr & 7) * 8 + (bit & 7));
    const uint64_t lo = w[0];
    if (sh == 0) return lo;
    return (lo >> sh) | (w[1] << (64 - sh));
}
ZD_HD uint8_t byte_at(const uint8_t *p, size_t i) { return p[i]; }
ZD_HD uint64_t le_at(const uint8_t *p, size_t i, int bytes) {  // bytes <= 8, byte loads only (headers, not hot)
    uint64_t v = 0;
    for (int k = 0; k < bytes; k++) v |= (uint64_t)p[i + k] << (8 * k);
    return v;
}
ZD_HD int highbit(uint32_t v) {  // index of the highest set bit, v != 0
#if defined(__CUDA_ARCH__)
    return 31 - __clz((int)v);
#else
    return 31 - __builtin_clz(v);
#endif
}

// backward bitstream (FSE / Huffman payloads): `pos` = number of bits not yet read; reading below bit 0 yields zeros.
// `c` holds the next `avail` unread bits left-aligned, so most reads touch no memory.
struct BackBits {
    const uint8_t *p;
    int64_t pos;
    uint64_t c;
    int avail;
    ZD_HD bool init(const uint8_t *base, size_t len) {
        p = base;
        c = 0;
        avail = 0;
        if (len == 0) return false;
        const uint8_t last = byte_at(base, len - 1);
        if (last == 0) return false;
        pos = (int64_t)(len - 1) * 8 + highbit(last);
        return true;
    }
};
ZD_HD uint32_t back_read(BackBits &b, int n) {  // n in [0, 32]
    if (n == 0) return 0;
    if (n > b.avail) {
        if (b.pos >= 64) b.c = window_at(b.p, (uint64_t)(b.pos - 64));
        else if (b.pos > 0) b.c = window_at(b.p, 0) << (64 - b.pos);
        else b.c = 0;
        b.avail = 64;
    }
    const uint32_t v = (uint32_t)(b.c >> (64 - n));
    b.c <<= n;
    b.avail -= n;
    b.pos -= n;
    return v;
}

// forward bitstream (FSE table descriptions)
struct FwdBits {
    const uint8_t *p;
    size_t len;
    uint64_t bit = 0;
};
ZD_HD uint32_t fwd_read(FwdBits &f, int n, bool *bad) {  // n <= 16
    if (f.bit + (uint64_t)n > (uint64_t)f.len * 8) {
        *bad = true;
        return 0;
    }
    const uint32_t v = (uint32_t)(window_at(f.p, f.bit) & ((1ull << n) - 1));
    f.bit += n;
    return v;
}

// ---------------------------------------------------------------- FSE tables
// reads a table description at src[0..len); fills norm[0..*nsym) and *log; returns bytes consumed, 0 on error
ZD_FN size_t fse_read_norm(const uint8_t *src, size_t len, int max_sym, int max_log, int16_t *norm, int *nsym, int *log) {
    FwdBits f{src, len};
    bool bad = false;
    const int al = 5 + (int)fwd_read(f, 4, &bad);
    if (bad || al > max_log) return 0;
    int remaining = 1 << al, sym = 0;
    while (remaining > 0 && sym <= max_sym) {
        const int bits = highbit((uint32_t)(remaining + 1)) + 1;
        uint32_t val = fwd_read(f, bits, &bad);
        if (bad) return 0;
        const uint32_t lower = (1u << (bits - 1)) - 1;
        const uint32_t threshold = (1u << bits) - 1 - (uint32_t)(remaining + 1);
        if ((val & lower) < threshold) {
            f.bit -= 1;
            val &= lower;
        } else if (val > lower) {
            val -= threshold;
        }
        const int proba = (int)val - 1;
        remaining -= proba < 0 ? -proba : proba;
        norm[sym++] = (int16_t)proba;
        if (proba == 0) {
            uint32_t rep = fwd_read(f, 2, &bad);
            for (;;) {
                if (bad) return 0;
                for (uint32_t i = 0; i < rep; i++) {
                    if (sym > max_sym) return 0;
                    norm[sym++] = 0;
                }
                if (rep != 3) break;
                rep = fwd_read(f, 2, &bad);
            }
        }
    }
    if (remaining != 0 || sym > max_sym + 1) return 0;
    *nsym = sym;
    *log = al;
    return (size_t)((f.bit + 7) / 8);
}

ZD_FN bool fse_build(const int16_t *norm, int nsym, int log, FseEntry *t, uint16_t *state_desc) {
    const int size = 1 << log;
    int high = size;
    for (int s = 0; s < nsym; s++)
        if (norm[s] == -1) {
            t[--high].sym = (uint8_t)s;
            state_desc[s] = 1;
        }
    const int step = (size >> 1) + (size >> 3) + 3, mask = size - 1;
    int pos = 0;
    for (int s = 0; s < nsym; s++) {
        if (norm[s] <= 0) continue;
        state_desc[s] = (uint16_t)norm[s];
        for (int i = 0; i < norm[s]; i++) {
            t[pos].sym = (uint8_t)s;
            do pos = (pos + step) & mask;
            while (pos >= high);
        }
    }
    if (pos != 0) return false;
    for (int i = 0; i < size; i++) {
        const uint16_t next = state_desc[t[i].sym]++;
        const int nb = log - highbit(next);
        t[i].nb = (uint8_t)nb;
        t[i].base = (uint16_t)(((uint32_t)next << nb) - (uint32_t)size);
    }
    return true;
}

// predefined distributions (RFC 8878 section 3.1.1.3.2.2), as arithmetic: no tables to index on the device
ZD_HD int16_t predef_ll(int i) {
    return i == 0 ? 4 : (i == 1 || i == 25) ? 3 : i >= 32 ? -1 : ((i >= 13 && i <= 15) || i >= 27) ? 1 : 2;
}
ZD_HD int16_t predef_ml(int i) { return i == 0 ? 1 : i == 1 ? 4 : i == 2 ? 3 : i <= 8 ? 2 : i <= 45 ? 1 : -1; }
ZD_HD int16_t predef_of(int i) { return (i >= 6 && i <= 8) ? 2 : i <= 23 ? 1 : -1; }

// literal-length / match-length code -> (base value, extra bits)  (RFC 8878 section 3.1.1.3.2.1.1)
ZD_HD int ll_bits(int c) { return c < 16 ? 0 : c < 20 ? 1 : c < 22 ? 2 : c < 24 ? 3 : c == 24 ? 4 : c == 25 ? 6 : c - 19; }
ZD_HD uint32_t ll_base(int c) {
    return c < 16 ? (uint32_t)c : c < 20 ? (uint32_t)(16 + 2 * (c - 16)) : c == 20 ? 24u : c == 21 ? 28u : c == 22 ? 32u : c == 23 ? 40u
           : c == 24 ? 48u : c == 25 ? 64u : 1u << (c - 19);
}
ZD_HD int ml_bits(int c) { return c < 32 ? 0 : c < 36 ? 1 : c < 38 ? 2 : c < 40 ? 3 : c < 42 ? 4 : c == 42 ? 5 : c == 43 ? 7 : c - 36; }
ZD_HD uint32_t ml_base(int c) {
    return c < 32 ? (uint32_t)(c + 3) : c < 36 ? (uint32_t)(35 + 2 * (c - 32)) : c == 36 ? 43u : c == 37 ? 47u : c == 38 ? 51u : c == 39 ? 59u
           : c == 40 ? 67u : c == 41 ? 83u : c == 42 ? 99u : c == 43 ? 131u : (1u << (c - 36)) + 3;
}
ZD_HD SeqEntry translate(FseEntry e, int which) {
    SeqEntry r;
    r.next_base = e.base;
    r.nb = e.nb;
    const int c = e.sym;
    r.add_bits = (uint8_t)(which == 0 ? ll_bits(c) : which == 1 ? c : ml_bits(c));
    r.base_value = which == 0 ? ll_base(c) : which == 1 ? 1u << c : ml_base(c);
    return r;
}

// one of the three sequence tables: mode 0 predefined, 1 RLE, 2 FSE description, 3 repeat.  Returns bytes consumed or -1
ZD_FN int seq_table(int mode, const uint8_t *src, size_t len, int which /*0 ll 1 of 2 ml*/, Work *w) {
    SeqEntry *t = which == 0 ? w->ll : which == 1 ? w->of : w->ml;
    int *log = which == 0 ? &w->ll_log : which == 1 ? &w->of_log : &w->ml_log;
    int *have = which == 0 ? &w->have_ll : which == 1 ? &w->have_of : &w->have_ml;
    const int max_sym = which == 0 ? kMaxLL : which == 1 ? kMaxOF : kMaxML;
    const int max_log = which == 1 ? 8 : 9;
    if (mode == 3) return *have ? 0 : -1;
    int used = 0, al = 0;
    if (mode == 1) {
        if (len < 1) return -1;
        const uint8_t s = byte_at(src, 0);
        if (s > max_sym) return -1;
        w->tmp[0].sym = s;
        w->tmp[0].nb = 0;
        w->tmp[0].base = 0;
        used = 1;
    } else {
        int nsym;
        if (mode == 0) {
            nsym = which == 0 ? 36 : which == 1 ? 29 : 53;
            for (int i = 0; i < nsym; i++) w->norm[i] = which == 0 ? predef_ll(i) : which == 1 ? predef_of(i) : predef_ml(i);
            al = which == 1 ? 5 : 6;
        } else {
            const size_t n = fse_read_norm(src, len, max_sym, max_log, w->norm, &nsym, &al);
            if (n == 0) return -1;
            used = (int)n;
        }
        if (!fse_build(w->norm, nsym, al, w->tmp, w->state_desc)) return -1;
    }
    for (int i = 0; i < (1 << al); i++) t[i] = translate(w->tmp[i], which);
    *log = al;
    *have = 1;
    return used;
}

// ---------------------------------------------------------------- Huffman literals
// tree description at src[0..len): fills w->huf / huf_log; returns bytes consumed, 0 on error
ZD_FN size_t huf_read_tree(const uint8_t *src, size_t len, Work *w) {
    if (len < 1) return 0;
    const int hb = byte_at(src, 0);
    int n = 0;
    size_t used;
    if (hb >= 128) {
        n = hb - 127;
        const size_t bytes = (size_t)(n + 1) / 2;
        if (1 + bytes > len) return 0;
        for (int i = 0; i < n; i++) {
            const uint8_t b = byte_at(src, 1 + (size_t)i / 2);
            w->weights[i] = (i & 1) ? (b & 15) : (b >> 4);
        }
        used = 1 + bytes;
    } else {
        if (hb == 0 || 1 + (size_t)hb > len) return 0;
        int nsym = 0, al = 0;
        const size_t hdr = fse_read_norm(src + 1, (size_t)hb, 12, 6, w->norm, &nsym, &al);
        if (hdr == 0 || hdr >= (size_t)hb) return 0;
        if (!fse_build(w->norm, nsym, al, w->wt, w->state_desc)) return 0;
        BackBits b;
        if (!b.init(src + 1 + hdr, (size_t)hb - hdr)) return 0;
        uint32_t s1 = back_read(b, al), s2 = back_read(b, al);
        if (b.pos < 0) return 0;
        for (;;) {
            if (n > 253) return 0;  // libzstd keeps room for two symbols per round; 255 weights at most
            w->weights[n++] = w->wt[s1].sym;
            s1 = w->wt[s1].base + back_read(b, w->wt[s1].nb);
            if (b.pos < 0) {
                w->weights[n++] = w->wt[s2].sym;
                break;
            }
            if (n > 253) return 0;
            w->weights[n++] = w->wt[s2].sym;
            s2 = w->wt[s2].base + back_read(b, w->wt[s2].nb);
            if (b.pos < 0) {
                w->weights[n++] = w->wt[s1].sym;
                break;
            }
        }
        used = 1 + (size_t)hb;
    }
    // the last weight is implied: the sum of 2^(w-1) must complete a power of two
    uint32_t sum = 0;
    for (int i = 0; i < n; i++) {
        if (w->weights[i] > kHufLogMax) return 0;
        if (w->weights[i]) sum += 1u << (w->weights[i] - 1);
    }
    if (sum == 0) return 0;
    const int max_bits = highbit(sum) + 1;
    if (max_bits > kHufLogMax) return 0;
    const uint32_t left = (1u << max_bits) - sum;
    if (left & (left - 1)) return 0;  // not a power of two
    w->weights[n++] = (uint8_t)(highbit(left) + 1);
    // table: codes are assigned by increasing weight (longest codes first), symbols in natural order inside a weight
    uint32_t rank_start[kHufLogMax + 2];
    uint32_t count[kHufLogMax + 2];
    for (int i = 0; i <= kHufLogMax + 1; i++) count[i] = 0;
    for (int i = 0; i < n; i++) count[w->weights[i]]++;
    if (count[1] < 2 || (count[1] & 1)) return 0;  // libzstd: at least two symbols of weight 1, and an even number
    uint32_t next = 0;
    for (int wt = 1; wt <= max_bits; wt++) {
        rank_start[wt] = next;
        next += count[wt] << (wt - 1);
    }
    if (next != (1u << max_bits)) return 0;
    for (int s = 0; s < n; s++) {
        const int wt = w->weights[s];
        if (!wt) continue;
        const uint32_t span = 1u << (wt - 1);
        const uint16_t e = (uint16_t)(s | ((max_bits + 1 - wt) << 8));
        for (uint32_t k = 0; k < span; k++) w->huf[rank_start[wt] + k] = e;
        rank_start[wt] += span;
    }
    w->huf_log = max_bits;
    w->have_huf = 1;
    return used;
}

// a sequence record: literal length (18 bits) | match length (18) | resolved offset (28)
ZD_HD uint64_t seq_pack(uint32_t ll, uint32_t ml, uint32_t offset) { return (uint64_t)ll | (uint64_t)ml << 18 | (uint64_t)offset << 36; }

}  // namespace zd
}  // namespace fheb
