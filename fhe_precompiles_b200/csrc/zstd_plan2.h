// Device zstd inflate (RFC 8878) up to the execution of the sequences (see zstd_dec.h for the contract: kZdOk means
// byte-identical to libzstd, anything else is handed back to the host).
//
// A frame's bitstreams are chains of dependent steps -- one GPU thread walks them at ~10x a host core's cost per step -- so
// throughput comes from (a) thousands of frames in flight and (b) splitting a frame into its INDEPENDENT chains and keeping
// each chain's inner loop to a few dozen instructions:
//   parse   one thread per frame   frame / block / section headers, Huffman and FSE table construction (per block, in global
//                                  scratch), descriptors of every bitstream                      (plan2_parse; k_zd2_parse)
//   huf     one thread per (frame, Huffman stream): the four literal streams of a block decode concurrently
//                                                                                                 (plan2_huf; k_zd3_huf)
//   seq     one lane per frame     FSE sequence chain -> (literal length, match length, resolved offset) records, with the
//                                  block's tables staged in shared memory                          (seq_block; k_zd3_seq)
// zstd_plan3.cuh executes the records (k_zd3_exec).  The bit readers use one aligned 32-bit load per 32 bits consumed and keep
// the unread bits left-aligned in a 64-bit register; the Huffman tables are read through the read-only path.
//
// The same source compiles for the host (tests/zd_host.cpp, compared with libzstd on fixtures, many levels and mutated frames)
// and for the device (codec_kernels.cu).
#pragma once
#include "zstd_dec.h"

namespace fheb {
namespace zd {

constexpr uint32_t kP2MaxBlocks = 4;       // a 131,169-byte ciphertext payload is two blocks; more go back to the host
constexpr uint32_t kP2MaxSeqs = 40960;

#if defined(__CUDA_ARCH__)
#define ZD_LDG32(p) __ldg((const unsigned int *)(p))
#define ZD_LDG16(p) __ldg((const unsigned short *)(p))
#else
#define ZD_LDG32(p) (*(const uint32_t *)(p))
#define ZD_LDG16(p) (*(const uint16_t *)(p))
#endif

struct Block2 {
    uint32_t type;             // 0 raw, 1 RLE, 2 compressed
    uint32_t src_off, size;    // raw: first byte / RLE: the byte; decompressed size
    uint32_t lit_mode;         // 0 raw literals inside src (lit_off), 1 RLE (lit_rle), 2 Huffman (decoded into lits + lit_off)
    uint32_t lit_off;
    int32_t lit_rle;
    uint32_t regen;
    uint32_t huf_tab, huf_log;        // Huffman table slot (the block that defined it) and its depth
    uint32_t nstreams;                // 1 or 4
    uint32_t st_off[4], st_len[4];    // stream bytes inside src
    uint32_t st_out[4], st_cnt[4];    // where its symbols go in lits, and how many
    uint32_t nseq, seq_off;           // records in seqs
    uint32_t bs_off, bs_len;          // sequence bitstream inside src
    uint32_t ll_tab, of_tab, ml_tab;  // table slots
    uint32_t ll_log, of_log, ml_log;
};
struct Plan2 {
    int32_t status;      // parse verdict; huf / seq downgrade it to kZdFallback through huf_bad / seq_bad
    int32_t huf_bad[4];  // one per stream thread (no atomics needed)
    int32_t seq_bad;
    uint32_t nblocks, content, window;
    Block2 blocks[kP2MaxBlocks];
};
struct Tables2 {  // per job: one slot per block
    uint16_t huf[kP2MaxBlocks][1 << kHufLogMax];
    SeqEntry ll[kP2MaxBlocks][512], of[kP2MaxBlocks][256], ml[kP2MaxBlocks][512];
};

// ---------------------------------------------------------------- backward bit reader, one aligned 32-bit load per refill
// The stream is src[0..len); its last byte's highest set bit is the end marker.  `c` holds the next unread bits left-aligned;
// `left` counts the stream bits not yet consumed (negative after an over-read; reads below bit 0 yield zeros).
struct Back32 {
    const uint32_t *wp;  // next word to load (descending)
    const uint32_t *w0;  // the aligned word that holds the first byte of the stream
    uint32_t lo_bits;    // bits of *w0 below the stream's first byte
    uint64_t c;
    int avail;
    int64_t left;
    ZD_HD bool init(const uint8_t *base, size_t len) {
        if (len == 0) return false;
        const uint8_t last = base[len - 1];
        if (last == 0) return false;
        const uintptr_t a = (uintptr_t)base;
        w0 = (const uint32_t *)(a & ~(uintptr_t)3);
        lo_bits = (uint32_t)(a & 3) * 8;
        left = (int64_t)(len - 1) * 8 + highbit(last);  // bits below the end marker
        const uint64_t abs_top = (uint64_t)lo_bits + (uint64_t)left;  // exclusive, in bits from *w0
        const uint32_t r = (uint32_t)(abs_top & 31);
        wp = w0 + (abs_top >> 5);
        c = 0;
        avail = 0;
        if (r) {
            uint32_t w = ZD_LDG32(wp) & ((1u << r) - 1);
            if (wp == w0 && lo_bits) w &= ~((1u << lo_bits) - 1);
            c = (uint64_t)w << (64 - r);
            avail = (int)r;
        }
        wp--;
        return true;
    }
    // afterwards avail >= 32 (bits below the stream read as zeros)
    ZD_HD void refill() {
        if (avail < 32) {
            uint32_t w = 0;
            if (wp >= w0) {
                w = ZD_LDG32(wp);
                if (wp == w0 && lo_bits) w &= ~((1u << lo_bits) - 1);
            }
            wp--;
            c |= (uint64_t)w << (32 - avail);
            avail += 32;
        }
    }
    ZD_HD uint32_t peek(int n) const { return (uint32_t)((c >> 1) >> (63 - n)); }  // n in [0, 32], n <= avail
    ZD_HD void skip(int n) {
        c <<= n;
        avail -= n;
        left -= n;
    }
    ZD_HD uint32_t read(int n) {
        const uint32_t v = peek(n);
        skip(n);
        return v;
    }
};

// ---------------------------------------------------------------- parse
// Every header and table of the frame, checked; the bitstreams are only located.  `w` is table-construction scratch.
ZD_FN int plan2_parse(const uint8_t *src, size_t slen, size_t cap, Work *w, Plan2 *plan, Tables2 *tabs) {
    plan->status = kZdFallback;
    plan->seq_bad = 0;
    for (int k = 0; k < 4; k++) plan->huf_bad[k] = 0;
    plan->nblocks = 0;
    if (slen < 6 || le_at(src, 0, 4) != 0xFD2FB528ull) return kZdFallback;
    const uint8_t fhd = byte_at(src, 4);
    const int fcs_flag = fhd >> 6, single = (fhd >> 5) & 1;
    if (fhd & 0x1F) return kZdFallback;
    size_t pos = 5, window = 0;
    if (!single) {
        if (pos >= slen) return kZdFallback;
        const uint8_t wd = byte_at(src, pos++);
        const int wlog = 10 + (wd >> 3);
        if (wlog > 27) return kZdFallback;
        window = ((size_t)1 << wlog) + (((size_t)1 << wlog) >> 3) * (wd & 7);
    }
    const int fcs_bytes = fcs_flag == 0 ? (single ? 1 : 0) : fcs_flag == 1 ? 2 : fcs_flag == 2 ? 4 : 8;
    if (fcs_bytes == 0 || pos + (size_t)fcs_bytes > slen) return kZdFallback;
    uint64_t fcs = le_at(src, pos, fcs_bytes);
    if (fcs_bytes == 2) fcs += 256;
    pos += (size_t)fcs_bytes;
    if (fcs > cap || fcs >= (1u << 27)) return kZdFallback;
    if (single) window = (size_t)fcs;
    const size_t block_max = window < kBlockMax ? window : kBlockMax;
    plan->content = (uint32_t)fcs;
    plan->window = (uint32_t)(window < (1u << 27) ? window : (1u << 27));
    w->have_ll = w->have_of = w->have_ml = w->have_huf = 0;
    uint32_t nblocks = 0, nseq_total = 0, lit_total = 0;
    uint32_t cur_huf = 0, cur_huf_log = 0, cur_ll = 0, cur_of = 0, cur_ml = 0;
    for (;;) {
        if (pos + 3 > slen || nblocks >= kP2MaxBlocks) return kZdFallback;
        const uint32_t bh = (uint32_t)le_at(src, pos, 3);
        pos += 3;
        const int last = bh & 1, type = (bh >> 1) & 3;
        const size_t bsize = bh >> 3;
        const uint32_t bi = nblocks++;
        Block2 &bp = plan->blocks[bi];
        bp.type = (uint32_t)type;
        bp.nseq = 0;
        bp.lit_mode = 0;
        bp.nstreams = 0;
        if (type == 3 || bsize > block_max) return kZdFallback;
        if (type == 0) {
            if (pos + bsize > slen) return kZdFallback;
            bp.src_off = (uint32_t)pos;
            bp.size = (uint32_t)bsize;
            pos += bsize;
        } else if (type == 1) {
            if (pos + 1 > slen) return kZdFallback;
            bp.src_off = (uint32_t)pos;
            bp.size = (uint32_t)bsize;
            pos += 1;
        } else {
            if (bsize < 2 || pos + bsize > slen) return kZdFallback;
            const uint8_t *b = src + pos;
            const size_t len = bsize;
            // ---- literals section
            const uint8_t b0 = byte_at(b, 0);
            const int ltype = b0 & 3, sf = (b0 >> 2) & 3;
            size_t hdr, regen, comp = 0;
            int streams = 1;
            if (ltype < 2) {
                hdr = (sf == 0 || sf == 2) ? 1 : sf == 1 ? 2 : 3;
                if (hdr > len) return kZdFallback;
                regen = hdr == 1 ? (size_t)(b0 >> 3) : (size_t)(le_at(b, 0, (int)hdr) >> 4);
                comp = ltype == 0 ? regen : 1;
            } else {
                hdr = sf <= 1 ? 3 : sf == 2 ? 4 : 5;
                if (hdr > len) return kZdFallback;
                const uint64_t v = le_at(b, 0, (int)hdr);
                const int bits = sf <= 1 ? 10 : sf == 2 ? 14 : 18;
                regen = (size_t)((v >> 4) & ((1u << bits) - 1));
                comp = (size_t)(v >> (4 + bits));
                streams = sf == 0 ? 1 : 4;
            }
            if (regen > block_max || hdr + comp > len) return kZdFallback;
            bp.regen = (uint32_t)regen;
            bp.lit_rle = -1;
            const uint8_t *lsrc = b + hdr;
            if (ltype == 0) {
                bp.lit_mode = 0;
                bp.lit_off = (uint32_t)(pos + hdr);
            } else if (ltype == 1) {
                bp.lit_mode = 1;
                bp.lit_rle = byte_at(lsrc, 0);
                bp.lit_off = 0;
            } else {
                if ((size_t)lit_total + regen > cap) return kZdFallback;
                size_t used = 0;
                if (ltype == 2) {
                    used = huf_read_tree(lsrc, comp, w);
                    if (used == 0) return kZdFallback;
                    cur_huf = bi;
                    cur_huf_log = (uint32_t)w->huf_log;
                    for (uint32_t k = 0; k < (1u << cur_huf_log); k++) tabs->huf[bi][k] = w->huf[k];
                } else if (!w->have_huf) {
                    return kZdFallback;
                }
                bp.lit_mode = 2;
                bp.huf_tab = cur_huf;
                bp.huf_log = cur_huf_log;
                bp.lit_off = lit_total;
                const size_t hoff = pos + hdr + used;  // first byte of the stream area inside src
                const uint8_t *hs = lsrc + used;
                const size_t hlen = comp - used;
                if (streams == 1) {
                    bp.nstreams = 1;
                    bp.st_off[0] = (uint32_t)hoff, bp.st_len[0] = (uint32_t)hlen;
                    bp.st_out[0] = lit_total, bp.st_cnt[0] = (uint32_t)regen;
                } else {
                    if (hlen < 6 + 4 || regen < 6) return kZdFallback;  // libzstd: >= 10 bytes and >= 6 literals for four streams
                    const size_t s1 = (size_t)le_at(hs, 0, 2), s2 = (size_t)le_at(hs, 2, 2), s3 = (size_t)le_at(hs, 4, 2);
                    const size_t seg = (regen + 3) / 4;
                    if (6 + s1 + s2 + s3 >= hlen || 3 * seg > regen) return kZdFallback;
                    const size_t s4 = hlen - 6 - s1 - s2 - s3;
                    const size_t lens[4] = {s1, s2, s3, s4};
                    bp.nstreams = 4;
                    size_t o = hoff + 6;
                    for (int k = 0; k < 4; k++) {
                        bp.st_off[k] = (uint32_t)o, bp.st_len[k] = (uint32_t)lens[k];
                        bp.st_out[k] = lit_total + (uint32_t)(k * seg);
                        bp.st_cnt[k] = (uint32_t)(k < 3 ? seg : regen - 3 * seg);
                        o += lens[k];
                    }
                }
                lit_total += (uint32_t)regen;
            }
            // ---- sequences section: count, table descriptions (built here), then the bitstream (decoded by seq_block)
            const uint8_t *ss = b + hdr + comp;
            const size_t sl = len - hdr - comp;
            if (sl < 1) return kZdFallback;
            size_t nseq = byte_at(ss, 0), sh = 1;
            if (nseq >= 128) {
                if (nseq == 255) {
                    if (sl < 3) return kZdFallback;
                    nseq = (size_t)le_at(ss, 1, 2) + 0x7F00;
                    sh = 3;
                } else {
                    if (sl < 2) return kZdFallback;
                    nseq = ((nseq - 128) << 8) + byte_at(ss, 1);
                    sh = 2;
                }
            }
            bp.nseq = (uint32_t)nseq;
            bp.seq_off = nseq_total;
            if (nseq == 0) {
                if (sl != 1) return kZdFallback;
            } else {
                if (nseq_total + nseq > kP2MaxSeqs || sl < sh + 1) return kZdFallback;
                const uint8_t modes = byte_at(ss, sh);
                if (modes & 3) return kZdFallback;
                size_t p = sh + 1;
                const int m_ll = modes >> 6, m_of = (modes >> 4) & 3, m_ml = (modes >> 2) & 3;
                // a table that this block defines is built straight into the block's slot; "repeat" keeps the previous slot
                if (m_ll != 3) w->ll = tabs->ll[bi], cur_ll = bi;
                if (m_of != 3) w->of = tabs->of[bi], cur_of = bi;
                if (m_ml != 3) w->ml = tabs->ml[bi], cur_ml = bi;
                int used = seq_table(m_ll, ss + p, sl - p, 0, w);
                if (used < 0) return kZdFallback;
                p += (size_t)used;
                if ((used = seq_table(m_of, ss + p, sl - p, 1, w)) < 0) return kZdFallback;
                p += (size_t)used;
                if ((used = seq_table(m_ml, ss + p, sl - p, 2, w)) < 0) return kZdFallback;
                p += (size_t)used;
                if (p >= sl) return kZdFallback;
                bp.ll_tab = cur_ll, bp.of_tab = cur_of, bp.ml_tab = cur_ml;
                bp.ll_log = (uint32_t)w->ll_log, bp.of_log = (uint32_t)w->of_log, bp.ml_log = (uint32_t)w->ml_log;
                bp.bs_off = (uint32_t)(pos + hdr + comp + p);
                bp.bs_len = (uint32_t)(sl - p);
                nseq_total += (uint32_t)nseq;
            }
            pos += bsize;
        }
        if (last) break;
    }
    if (pos != slen) return kZdFallback;
    plan->nblocks = nblocks;
    plan->status = kZdOk;
    return kZdOk;
}

// ---------------------------------------------------------------- Huffman streams
// stream `k` (0..3) of every Huffman block of the frame; false unless each stream is consumed exactly
ZD_FN bool plan2_huf(const uint8_t *src, const Plan2 *plan, const Tables2 *tabs, uint8_t *lits, int k) {
    if (plan->status != kZdOk) return true;
    for (uint32_t bi = 0; bi < plan->nblocks; bi++) {
        const Block2 &bp = plan->blocks[bi];
        if (bp.type != 2 || bp.lit_mode != 2 || (uint32_t)k >= bp.nstreams) continue;
        Back32 b;
        if (!b.init(src + bp.st_off[k], bp.st_len[k])) return false;
        const uint16_t *tab = tabs->huf[bp.huf_tab];
        const int log = (int)bp.huf_log;
        uint8_t *out = lits + bp.st_out[k];
        const uint32_t count = bp.st_cnt[k];
        // eight symbols per 64-bit store where the destination allows: byte stores from one thread are what is slow
        uint32_t i = 0;
        for (; i < count && (((uintptr_t)(out + i)) & 7); i++) {
            b.refill();
            const uint32_t e = ZD_LDG16(tab + b.peek(log));
            out[i] = (uint8_t)e;
            b.skip((int)(e >> 8));
        }
        for (; i + 8 <= count; i += 8) {
            uint64_t pack = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                b.refill();
                const uint32_t e = ZD_LDG16(tab + b.peek(log));
                pack |= (uint64_t)(e & 0xFF) << (8 * j);
                b.skip((int)(e >> 8));
            }
            *(uint64_t *)(out + i) = pack;
        }
        for (; i < count; i++) {
            b.refill();
            const uint32_t e = ZD_LDG16(tab + b.peek(log));
            out[i] = (uint8_t)e;
            b.skip((int)(e >> 8));
        }
        if (b.left != 0) return false;
    }
    return true;
}

// ---------------------------------------------------------------- sequences
// The FSE sequence chain of a block, as k_zd3_seq runs it (zstd_plan3.cuh seq_frames stages the tables and calls seq_block).
constexpr int kTabCells = 512 + 256 + 512;  // LL (log <= 9), OF (<= 8), ML (<= 9)
constexpr int kLutCells = 36 + 53;          // base values of the literal-length and match-length codes (one copy per CTA)

// A table cell in shared memory: next state base (10 bits) | state bits << 10 (4) | value bits << 14 (5) | code << 19 (6).  The
// value's BASE is a function of the code alone (RFC 8878 3.1.1.3.2.1.1) and is not on the chain that links one sequence to the
// next - only the bit counts are - so it comes from a small per-CTA table after the fact and a cell is 4 bytes instead of 8.
static_assert(sizeof(SeqEntry) == 8, "SeqEntry is read as one 8-byte cell");
ZD_HD uint32_t pack_cell(uint2 g, int which) {  // g: a SeqEntry as stored by the parse step
    const uint32_t next_base = g.x & 0xFFFF, nb = (g.x >> 16) & 0xFF, add = g.x >> 24, base = g.y;
    uint32_t code;
    if (which == 1) {
        code = add;  // offset code: base = 1 << code
    } else if (which == 0) {
        code = add == 0 ? base : add == 1 ? 16 + (base - 16) / 2 : add == 2 ? 20 + (base - 24) / 4 : add == 3 ? 22 + (base - 32) / 8
               : add == 4 ? 24u : add == 6 ? 25u : add + 19;
    } else {
        code = add == 0 ? base - 3 : add == 1 ? 32 + (base - 35) / 2 : add == 2 ? 36 + (base - 43) / 4 : add == 3 ? 38 + (base - 51) / 8
               : add == 4 ? 40 + (base - 67) / 16 : add == 5 ? 42u : add == 7 ? 43u : add + 36;
    }
    return next_base | nb << 10 | add << 14 | (code & 63) << 19;
}

// PTX shifts clamp at 32: a shift by 32 yields 0.  The host must do the same (x86 would shift by n mod 32).
ZD_HD uint32_t shl32(uint32_t v, uint32_t n) {
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(n));
    return r;
#else
    return n >= 32 ? 0u : v << n;
#endif
}
ZD_HD uint32_t shr32(uint32_t v, uint32_t n) {
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("shr.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(n));
    return r;
#else
    return n >= 32 ? 0u : v >> n;
#endif
}

// backward bit reader on aligned 32-bit words (Back32) with the next word already in a register
struct Back32P {
    const uint32_t *wp, *w0;
    uint32_t lo_bits, nextw, nextmask;  // the prefetched word is masked when it is CONSUMED: nothing waits for the load before
    uint64_t c;   // unread bits, left-aligned
    int avail;    // how many of them are valid
    int left;     // stream bits not yet consumed (negative after an over-read; a stream is < 2^20 bits)
    ZD_HD void fetch() {
        nextw = 0, nextmask = 0;
        if (wp >= w0) {
            nextw = ZD_LDG32(wp);
            nextmask = wp == w0 ? ~((1u << lo_bits) - 1) : 0xFFFFFFFFu;
        }
    }
    ZD_HD bool init(const uint8_t *base, size_t len) {
        if (len == 0 || len > (1u << 17)) return false;
        const uint8_t last = base[len - 1];
        if (last == 0) return false;
        const uintptr_t a = (uintptr_t)base;
        w0 = (const uint32_t *)(a & ~(uintptr_t)3);
        lo_bits = (uint32_t)(a & 3) * 8;
        left = (int)(len - 1) * 8 + highbit(last);
        const uint32_t abs_top = lo_bits + (uint32_t)left;
        const uint32_t r = abs_top & 31;
        wp = w0 + (abs_top >> 5);
        c = 0;
        avail = 0;
        if (r) {
            uint32_t w = ZD_LDG32(wp) & ((1u << r) - 1);
            if (wp == w0 && lo_bits) w &= ~((1u << lo_bits) - 1);
            c = (uint64_t)w << (64 - r);
            avail = (int)r;
        }
        wp--;
        fetch();
        return true;
    }
    ZD_HD void refill() {  // afterwards avail >= 32
        if (avail < 32) {
            c |= (uint64_t)(nextw & nextmask) << (32 - avail);
            avail += 32;
            wp--;
            fetch();
        }
    }
    ZD_HD uint32_t read(int n) {  // n in [0, 32], n <= avail
        const uint32_t v = (uint32_t)((c >> 1) >> (63 - n));
        c <<= n;
        avail -= n;
        left -= n;
        return v;
    }
};

// The sequences of one block -> (literal length, match length, resolved offset) records at `so`, and the block's verdict.  The
// per-sequence checks are monotone (bits left, literal total) or independent of the other sequences (value ranges), so they are
// accumulated and judged once after the loop; a sequence whose six bit fields fit the 32 bits a single refill guarantees - all
// but a handful - takes them from one register.  The repeat offsets r0_, r1_, r2_ carry over from one block to the next.
ZD_HD bool seq_block(const uint8_t *src, const Block2 &bp, const uint32_t *tll, const uint32_t *tof, const uint32_t *tml,
                     const uint32_t *lut, uint64_t *so, uint32_t &r0_, uint32_t &r1_, uint32_t &r2_) {
    Back32P b;
    if (!b.init(src + bp.bs_off, bp.bs_len)) return false;
    b.refill();
    uint32_t st_ll = b.read((int)bp.ll_log), st_of = b.read((int)bp.of_log), st_ml = b.read((int)bp.ml_log);
    if (b.left < 0) return false;
    const uint32_t nseq = bp.nseq, regen = bp.regen;
    uint32_t r0 = r0_, r1 = r1_, r2 = r2_;
    uint32_t lsum = 0, badacc = 0;  // (lsum: < 2^18 per term, < 2^16 terms)
    for (uint32_t i = 0; i < nseq; i++) {
        const uint32_t el = tll[st_ll], eo = tof[st_of], em = tml[st_ml];
        const uint32_t keep = i + 1 < nseq ? 0xFu : 0u;  // the last sequence reads no state bits
        const uint32_t a_of = (eo >> 14) & 31, a_ml = (em >> 14) & 31, a_ll = (el >> 14) & 31;
        const uint32_t n_ll = (el >> 10) & keep, n_ml = (em >> 10) & keep, n_of = (eo >> 10) & keep;
        const uint32_t s1 = a_of + a_ml, s2 = s1 + a_ll, s3 = s2 + n_ll, s4 = s3 + n_ml, tot = s4 + n_of;
        uint32_t x_of, x_ml, x_ll, y_ll, y_ml, y_of;
        b.refill();
        if (tot <= 32) {
            const uint32_t hi = (uint32_t)(b.c >> 32);
            x_of = shr32(hi, 32 - a_of);
            x_ml = shr32(shl32(hi, a_of), 32 - a_ml);
            x_ll = shr32(shl32(hi, s1), 32 - a_ll);
            y_ll = shr32(shl32(hi, s2), 32 - n_ll);
            y_ml = shr32(shl32(hi, s3), 32 - n_ml);
            y_of = shr32(shl32(hi, s4), 32 - n_of);
            b.c <<= tot;
            b.avail -= (int)tot;
            b.left -= (int)tot;
        } else {
            x_of = b.read((int)a_of);
            b.refill();
            x_ml = b.read((int)a_ml);
            x_ll = b.read((int)a_ll);
            b.refill();
            y_ll = b.read((int)n_ll);
            y_ml = b.read((int)n_ml);
            y_of = b.read((int)n_of);
        }
        st_ll = (el & 0x3FF) + y_ll;
        st_ml = (em & 0x3FF) + y_ml;
        st_of = (eo & 0x3FF) + y_of;
        const uint32_t ofv = (1u << a_of) + x_of, ml = lut[36 + (em >> 19)] + x_ml, ll = lut[el >> 19] + x_ll;
        uint32_t offset;
        if (ofv > 3) {
            offset = ofv - 3;
            r2 = r1, r1 = r0, r0 = offset;
        } else {
            const uint32_t idx = ofv - 1 + (ll == 0 ? 1 : 0);
            if (idx == 0) {
                offset = r0;
            } else {
                if (idx == 3 && r0 == 1) return false;  // offset 0: libzstd patches it up; let it decide
                offset = idx == 1 ? r1 : idx == 2 ? r2 : r0 - 1;
                if (idx != 1) r2 = r1;
                r1 = r0, r0 = offset;
            }
        }
        lsum += ll;
        badacc |= (offset >> 27) | ((ll | ml) >> 18) | (lsum >> 30);
        so[i] = seq_pack(ll & 0x3FFFF, ml & 0x3FFFF, offset);
    }
    r0_ = r0, r1_ = r1, r2_ = r2;
    return b.left == 0 && badacc == 0 && lsum <= regen;
}

}  // namespace zd
}  // namespace fheb
