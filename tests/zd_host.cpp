// Host build of the device zstd decoder (fhe_precompiles_b200/csrc: zstd_dec.h, zstd_plan2.h, zstd_exec3.h) for
// tests/test_zstd_dec.py: the same source that k_zd2_parse, k_zd3_huf, k_zd3_seq and k_zd3_exec run, compiled with g++ so that
// it can be compared with libzstd and fuzzed without a GPU.  Where a kernel spreads a step over many threads, the threads are
// played one after the other between the kernel's barriers.
#include <algorithm>
#include <cstring>
#include <vector>

#include "zstd_exec3.h"
#include "zstd_plan2.h"

// parse -> Huffman streams -> sequence chains -> execution.  *rounds = jump rounds of the busiest pass of the execution, *polls =
// the number of times a thread found its source still pending in its step 3 (0 when the jumping resolved everything).
extern "C" int zd_decode(const uint8_t *src, size_t slen, uint8_t *dst, size_t cap, size_t *dlen, int *rounds, long *polls) {
    using namespace fheb::zd;
    using namespace fheb::zd3;
    static thread_local Work *w = nullptr;
    static thread_local Plan2 *plan = nullptr;
    static thread_local Tables2 *tabs = nullptr;
    static thread_local std::vector<uint64_t> seqs(kP2MaxSeqs);
    if (!w) {
        w = new Work();
        plan = new Plan2();
        tabs = new Tables2();
    }
    work_bind(w, nullptr);
    std::vector<uint8_t> buf(slen + 2 * kPad + 8, 0xAA), lits(cap + 16);
    uint8_t *f = buf.data() + kPad + 3;
    memcpy(f, src, slen);
    if (rounds) *rounds = 0;
    if (polls) *polls = 0;
    if (plan2_parse(f, slen, cap, w, plan, tabs) != kZdOk) return 1;
    for (int k = 0; k < 4; k++)
        if (!plan2_huf(f, plan, tabs, lits.data(), k)) return 1;
    {  // k_zd3_seq (zstd_plan3.cuh seq_frames) for one frame slot
        std::vector<uint32_t> tab(kTabCells), lut(kLutCells);
        for (int c = 0; c < kLutCells; c++) lut[c] = c < 36 ? ll_base(c) : ml_base(c - 36);
        const auto stage = [](uint32_t *dst, const SeqEntry *src, uint32_t log, int which) {
            for (uint32_t k = 0; k < (1u << log); k++) {
                uint2 g;  // the device's 8-byte load of a cell
                memcpy(&g, src + k, sizeof g);
                dst[k] = pack_cell(g, which);
            }
        };
        uint32_t r0 = 1, r1 = 4, r2 = 8;
        for (uint32_t bi = 0; bi < plan->nblocks; bi++) {
            const Block2 &bp = plan->blocks[bi];
            if (bp.type != 2 || bp.nseq == 0) continue;
            if (bp.ll_log > 9 || bp.of_log > 8 || bp.ml_log > 9) return 1;
            stage(tab.data(), tabs->ll[bp.ll_tab], bp.ll_log, 0);
            stage(tab.data() + 512, tabs->of[bp.of_tab], bp.of_log, 1);
            stage(tab.data() + 768, tabs->ml[bp.ml_tab], bp.ml_log, 2);
            if (!seq_block(f, bp, tab.data(), tab.data() + 512, tab.data() + 768, lut.data(), seqs.data() + bp.seq_off, r0, r1, r2))
                return 1;
        }
    }
    if (plan->content > kExecOutBytes - 31) return 1;
    const int T = kExecThreads;
    std::vector<uint8_t> out(kExecOutBytes, 0xEE);
    std::vector<uint32_t> pend(kExecBitWords, 0), start(kExecBitWords, 0);
    const uint32_t content = plan->content, window = plan->window;
    const uint32_t block_max = window < kBlockMax ? window : (uint32_t)kBlockMax;
    uint32_t pos = 0;
    for (uint32_t bi = 0; bi < plan->nblocks; bi++) {
        const Block2 &bp = plan->blocks[bi];
        if (bp.type != 2) {
            if (bp.size > content - pos) return 1;
            for (uint32_t k = 0; k < bp.size; k++) out[pos + k] = bp.type == 0 ? f[bp.src_off + k] : f[bp.src_off];
            pos += bp.size;
            continue;
        }
        const uint8_t *lit = bp.lit_mode == 0 ? f + bp.lit_off : lits.data() + bp.lit_off;
        const int lit_rle = bp.lit_mode == 1 ? bp.lit_rle : -1;
        const uint32_t nseq = bp.nseq, regen = bp.regen;
        uint64_t *so = seqs.data() + bp.seq_off;
        const uint32_t per = (nseq + T - 1) / T;
        std::vector<uint64_t> ex_ll(T), ex_o(T);
        uint64_t tot_ll = 0, tot_o = 0;
        for (int t = 0; t < T; t++) {
            const uint32_t lo = std::min((uint32_t)t * per, nseq), hi = std::min(lo + per, nseq);
            ex_ll[t] = tot_ll, ex_o[t] = tot_o;
            for (uint32_t i = lo; i < hi; i++) {
                const uint32_t ll = (uint32_t)(so[i] & 0x3FFFF), ml = (uint32_t)((so[i] >> 18) & 0x3FFFF);
                tot_ll += ll, tot_o += (uint64_t)ll + ml;
            }
        }
        if (tot_ll > regen) return 1;
        const uint64_t total_out = tot_o + (regen - tot_ll);
        if (total_out > (uint64_t)(content - pos) || total_out > block_max) return 1;
        bool ok = true;
        for (int t = 0; t < T; t++) {
            const uint32_t lo = std::min((uint32_t)t * per, nseq), hi = std::min(lo + per, nseq);
            ok &= place_sequences(so, lo, hi, (uint32_t)ex_ll[t], pos + (uint32_t)ex_o[t], lit, lit_rle, window, out.data(), pend.data(),
                                  start.data());
        }
        for (uint32_t k = 0; k < regen - (uint32_t)tot_ll; k++)
            out[pos + (uint32_t)tot_o + k] = lit_rle >= 0 ? (uint8_t)lit_rle : lit[(uint32_t)tot_ll + k];
        if (!ok) return 1;
        for (uint32_t cbase = 0; cbase < nseq; cbase += kExecChunk) {
            std::vector<uint32_t> F((size_t)T * kExecPer, 0), MI((size_t)T * kExecPer, 0), act(T, 0), chg(T, 0);
            for (int t = 0; t < T; t++)
                for (int k = 0; k < kExecPer; k++) {
                    const uint32_t i = cbase + (uint32_t)k * T + t;
                    if (i < nseq && jump_init(so[i], &F[t * kExecPer + k], &MI[t * kExecPer + k])) act[t] |= 1u << k;
                }
            const uint32_t stop_below = std::min(nseq - cbase, kExecChunk) / kExecStopShare;
            for (int round = 0; round < kExecMaxRounds; round++) {
                bool any = false;
                uint32_t moved = 0;
                for (int t = 0; t < T; t++) {
                    chg[t] = 0;
                    for (int k = 0; k < kExecPer; k++) {
                        if (!((act[t] >> k) & 1)) continue;
                        const int r = jump_look(pend.data(), start.data(), out.data(), &F[t * kExecPer + k], &MI[t * kExecPer + k],
                                                so + cbase + (uint32_t)k * T + t);
                        if (r == kJumpStop) {
                            act[t] &= ~(1u << k);
                            continue;
                        }
                        moved++;
                        if (r == kJumpPublish) chg[t] |= 1u << k;
                        else chg[t] |= 1u << 16;
                    }
                    any |= chg[t] != 0;
                }
                for (int t = 0; t < T; t++)
                    for (int k = 0; k < kExecPer; k++)
                        if ((chg[t] >> k) & 1) jump_publish(out.data(), F[t * kExecPer + k], MI[t * kExecPer + k]);
                if (rounds && round + 1 > *rounds) *rounds = round + 1;
                if (!any || moved < stop_below) break;
            }
            // step 3: warps of 32 threads, each polling until its current 32 matches are copied; the warps take turns
            std::vector<int> kcur(T / 32, 0);
            std::vector<std::vector<char>> waiting(T / 32, std::vector<char>(32, 0));
            std::vector<std::vector<CopyJob>> jobs(T / 32, std::vector<CopyJob>(32));
            auto load = [&](int wp) {
                for (int l = 0; l < 32; l++) {
                    const int t = wp * 32 + l, k = kcur[wp];
                    const uint32_t i = cbase + (uint32_t)k * T + t;
                    jobs[wp][l] = copy_job(i < nseq ? so[i] : 0, F[t * kExecPer + k], MI[t * kExecPer + k]);
                    waiting[wp][l] = jobs[wp][l].ml != 0;
                }
            };
            for (int wp = 0; wp < T / 32; wp++) load(wp);
            for (bool busy = true; busy;) {
                busy = false;
                bool progress = false;
                for (int wp = 0; wp < T / 32; wp++) {
                    if (kcur[wp] >= kExecPer) continue;
                    busy = true;
                    bool any_wait = false;
                    for (int l = 0; l < 32; l++) {
                        if (!waiting[wp][l]) continue;
                        if (copy_ready(pend.data(), jobs[wp][l])) {
                            copy_match(out.data(), jobs[wp][l]);
                            pend_clear(pend.data(), jobs[wp][l].m, jobs[wp][l].ml);
                            waiting[wp][l] = 0;
                            progress = true;
                        } else {
                            any_wait = true;
                            if (polls) ++*polls;
                        }
                    }
                    if (!any_wait) {
                        progress = true;
                        if (++kcur[wp] < kExecPer) load(wp);
                    }
                }
                if (busy && !progress) return 2;  // a deadlock would hang the kernel: fail the test instead
            }
        }
        pos += (uint32_t)total_out;
    }
    if (pos != content) return 1;
    memcpy(dst, out.data(), content);
    *dlen = content;
    return 0;
}
