// Device zstd inflate: the sequence chains and the execution, after zstd_plan2.h's parse and Huffman steps (device-only; same
// contract as zstd_dec.h: kJobOk means byte-identical to libzstd, everything else goes back to the host).
//
// Measured on level-3 ciphertext frames (raw literals, 16,354 sequences of ~4 literal + ~4 match bytes, three 512/256/512-cell
// FSE tables per frame), a thread per frame for both steps (profiles/r2_codec.md) leaves two things on the table:
//   * a sequence chain that reads its FSE tables from global memory at 0.5 MB per lane stride makes three dependent L2 round
//     trips per sequence, with 32 frames diverging inside one warp;
//   * execution by one THREAD per frame runs 16 k sequences one after the other although only the match copies depend on each other.
// Here:
//   k_zd3_seq   four frames per warp (a one-lane warp costs as many issue slots as a full one, and shared memory - 5 KB of FSE
//               tables per frame as 4-byte cells - bounds the frames per SM either way): each frame's tables are staged in shared
//               memory, the bit reader keeps the next stream word prefetched, a sequence's six bit fields come out of one register
//               (zstd_plan2.h seq_block)
//   k_zd3_exec  one CTA (1,024 threads) per frame, the frame's output assembled in shared memory: prefix sums give every
//               sequence its literal and output positions, literals are copied in parallel, pointer jumping moves every match's
//               source back along its chain of pending matches (zstd_exec3.h), and the copies go through a per-byte "pending"
//               bitmap (a match is copied once none of its source bytes is pending; dependencies point backwards only, so the
//               earliest pending match is always ready); the payload leaves with 16-byte stores
#pragma once
#include "codec_kernels.h"
#include "zstd_plan2.h"

namespace fheb {
namespace zd3 {

using zd::Block2;
using zd::Plan2;
using zd::Tables2;

constexpr int kSeqFrames = 4;  // frames per warp of k_zd3_seq: lanes 0, 8, 16, 24 walk one chain each
constexpr size_t kSeqSmem = ((size_t)kSeqFrames * zd::kTabCells + zd::kLutCells) * sizeof(uint32_t);  // 20.4 KB per one-warp CTA: 11 CTAs per SM

// One warp, up to kSeqFrames frames: slot s = lane / 8; its eight lanes stage the block's tables, lane 8 s walks the chain.
// `tabs_smem`: kSeqFrames x kTabCells cells, then the kLutCells base values.  Returns the slot's verdict to its eight lanes.
__device__ __forceinline__ bool seq_frames(const uint8_t *src, const Plan2 *plan, const Tables2 *tabs, uint64_t *seqs, bool have,
                                           uint32_t *tabs_smem) {
    const int lane = threadIdx.x & 31, sub = lane & 7;
    uint32_t *T = tabs_smem + (size_t)(lane >> 3) * zd::kTabCells;
    uint32_t *lut = tabs_smem + (size_t)kSeqFrames * zd::kTabCells;
    for (int c = lane; c < zd::kLutCells; c += 32) lut[c] = c < 36 ? zd::ll_base(c) : zd::ml_base(c - 36);
    uint32_t r0 = 1, r1 = 4, r2 = 8;
    bool ok = have;
    for (uint32_t bi = 0; bi < zd::kP2MaxBlocks; bi++) {
        const Block2 *bp = have && bi < plan->nblocks ? &plan->blocks[bi] : nullptr;
        const bool run = ok && bp && bp->type == 2 && bp->nseq != 0;
        __syncwarp();
        if (run) {
            if (bp->ll_log > 9 || bp->of_log > 8 || bp->ml_log > 9) {
                ok = false;
            } else {
                const uint2 *gll = (const uint2 *)tabs->ll[bp->ll_tab], *gof = (const uint2 *)tabs->of[bp->of_tab],
                            *gml = (const uint2 *)tabs->ml[bp->ml_tab];
                for (uint32_t k = sub; k < (1u << bp->ll_log); k += 8) T[k] = zd::pack_cell(__ldg(gll + k), 0);
                for (uint32_t k = sub; k < (1u << bp->of_log); k += 8) T[512 + k] = zd::pack_cell(__ldg(gof + k), 1);
                for (uint32_t k = sub; k < (1u << bp->ml_log); k += 8) T[768 + k] = zd::pack_cell(__ldg(gml + k), 2);
            }
        }
        __syncwarp();
        if (run && ok && sub == 0) ok = zd::seq_block(src, *bp, T, T + 512, T + 768, lut, seqs + bp->seq_off, r0, r1, r2);
        ok = __shfl_sync(0xFFFFFFFFu, (int)ok, lane & ~7) != 0;
    }
    return ok;
}

}  // namespace zd3
}  // namespace fheb

#include "zstd_exec3.h"
static_assert(fheb::zd3::kExecOutBytes == fheb::kPayloadStride, "the output buffer is one payload slot");

namespace fheb {
namespace zd3 {

// block-wide exclusive scan of one 64-bit value per thread (kExecThreads threads); *total = the sum.  `tmp`: 33 words.
__device__ __forceinline__ uint64_t block_exscan(uint64_t v, uint64_t *tmp, uint64_t *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint64_t o = __shfl_up_sync(0xFFFFFFFFu, inc, d);
        if (lane >= d) inc += o;
    }
    __syncthreads();  // tmp may still be read from a previous call
    if (lane == 31) tmp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const uint64_t w = tmp[lane];
        uint64_t winc = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint64_t o = __shfl_up_sync(0xFFFFFFFFu, winc, d);
            if (lane >= d) winc += o;
        }
        tmp[lane] = winc - w;
        if (lane == 31) tmp[32] = winc;
    }
    __syncthreads();
    *total = tmp[32];
    return tmp[warp] + inc - v;
}

// Executes the plan of one frame with the whole CTA (the steps are described in zstd_exec3.h).  `seqs` is rewritten in place.
// Returns kZdOk with the payload in dst[0, content) (dst: 16-byte aligned, kPayloadStride bytes), else kZdFallback.
__device__ __forceinline__ int exec_frame(const uint8_t *src, const Plan2 *plan, uint64_t *seqs, const uint8_t *lits, uint8_t *dst,
                                          uint8_t *smem) {
    uint8_t *out = smem;
    uint32_t *pend = (uint32_t *)(smem + kExecOutBytes);
    uint32_t *start = pend + kExecBitWords;
    uint64_t *tmp = (uint64_t *)(start + kExecBitWords);
    int *bad = (int *)(tmp + 64);
    uint32_t *moved_cnt = (uint32_t *)(tmp + 64) + 2;  // matches moved in a jump round (two alternating counters)
    uint8_t *lit_smem = (uint8_t *)(tmp + 64) + 64;
    const int t = threadIdx.x;
    if (t == 0) *bad = 0;
    for (uint32_t k = t; k < 2 * kExecBitWords; k += kExecThreads) pend[k] = 0;  // both bitmaps
    __syncthreads();
    const uint32_t cap = plan->content, window = plan->window;
    const uint32_t block_max = window < zd::kBlockMax ? window : (uint32_t)zd::kBlockMax;
    if (cap > kCtPayloadBytes) return zd::kZdFallback;
    uint32_t pos = 0;  // uniform
    const uint32_t nblocks = plan->nblocks;
    for (uint32_t bi = 0; bi < nblocks; bi++) {
        const Block2 &bp = plan->blocks[bi];
        if (bp.type != 2) {
            if (bp.size > cap - pos) return zd::kZdFallback;
            if (bp.type == 0) {
                const uint8_t *s = src + bp.src_off;
                for (uint32_t k = t; k < bp.size; k += kExecThreads) out[pos + k] = s[k];
            } else {
                const uint8_t v = src[bp.src_off];
                for (uint32_t k = t; k < bp.size; k += kExecThreads) out[pos + k] = v;
            }
            pos += bp.size;
            __syncthreads();
            continue;
        }
        const uint8_t *lit = bp.lit_mode == 0 ? src + bp.lit_off : lits + bp.lit_off;
        const int lit_rle = bp.lit_mode == 1 ? bp.lit_rle : -1;
        const uint32_t nseq = bp.nseq, regen = bp.regen;
        uint64_t *so = seqs + bp.seq_off;
        if (kExecLitBytes && lit_rle < 0 && regen <= kExecLitBytes) {  // (the barriers of the scans below order these stores before their readers)
            for (uint32_t k = t; k < regen; k += kExecThreads) lit_smem[k] = lit[k];
            lit = lit_smem;
        }
        // ---- 1 positions: warp w owns a run of consecutive sequences, lane l its sequences l, l + 32, ...: neighbouring lanes
        // work on neighbouring sequences, so their records load coalesced and their output bytes fall in different banks
        // (16 consecutive sequences per THREAD put every lane of a warp 128 bytes apart: 32-way conflicts on each store)
        const int lane = t & 31, warp = t >> 5;
        const uint32_t rows = ((nseq + 31) / 32 + 31) / 32;  // rows of 32 sequences per warp
        const uint32_t wlo = min((uint32_t)warp * rows * 32, nseq), whi = min(wlo + rows * 32, nseq);
        uint64_t s_ll = 0, s_o = 0;
        for (uint32_t i = wlo + lane; i < whi; i += 32) {
            const uint64_t e = so[i];
            const uint32_t ll = (uint32_t)(e & 0x3FFFF), ml = (uint32_t)((e >> 18) & 0x3FFFF);
            s_ll += ll;
            s_o += (uint64_t)ll + ml;
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            s_ll += __shfl_xor_sync(0xFFFFFFFFu, s_ll, d);
            s_o += __shfl_xor_sync(0xFFFFFFFFu, s_o, d);
        }
        uint64_t tot_ll, tot_o;
        uint64_t run_ll = block_exscan(lane == 0 ? s_ll : 0, tmp, &tot_ll);  // lane 0: the sum over the warps before this one
        uint64_t run_o = block_exscan(lane == 0 ? s_o : 0, tmp, &tot_o);
        run_ll = __shfl_sync(0xFFFFFFFFu, run_ll, 0);
        run_o = __shfl_sync(0xFFFFFFFFu, run_o, 0);
        if (tot_ll > regen) return zd::kZdFallback;  // (uniform: the totals are)
        const uint64_t total_out = tot_o + (regen - tot_ll);
        if (total_out > (uint64_t)(cap - pos) || total_out > block_max) return zd::kZdFallback;
        {
            bool ok = true;
            for (uint32_t r0 = wlo; r0 < whi; r0 += 32) {  // (uniform per warp)
                const uint32_t i = r0 + lane;
                uint32_t ll = 0, both = 0;
                if (i < whi) {
                    const uint64_t e = so[i];
                    ll = (uint32_t)(e & 0x3FFFF);
                    both = ll + (uint32_t)((e >> 18) & 0x3FFFF);
                }
                uint32_t inc_ll = ll, inc_o = both;  // (a row's totals fit 32 bits: 32 x 2^19)
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t a_ = __shfl_up_sync(0xFFFFFFFFu, inc_ll, d), b_ = __shfl_up_sync(0xFFFFFFFFu, inc_o, d);
                    if (lane >= d) inc_ll += a_, inc_o += b_;
                }
                if (i < whi)
                    ok &= place_sequences(so, i, i + 1, (uint32_t)run_ll + inc_ll - ll, pos + (uint32_t)run_o + inc_o - both, lit, lit_rle,
                                          window, out, pend, start);
                run_ll += __shfl_sync(0xFFFFFFFFu, inc_ll, 31);
                run_o += __shfl_sync(0xFFFFFFFFu, inc_o, 31);
            }
            if (!ok) *bad = 1;
        }
        {
            const uint32_t tail = regen - (uint32_t)tot_ll, tpos = pos + (uint32_t)tot_o;
            if (lit_rle >= 0) {
                for (uint32_t k = t; k < tail; k += kExecThreads) out[tpos + k] = (uint8_t)lit_rle;
            } else {
                for (uint32_t k = t; k < tail; k += kExecThreads) out[tpos + k] = lit[(uint32_t)tot_ll + k];
            }
        }
        __syncthreads();
        if (*bad) return zd::kZdFallback;
        for (uint32_t cbase = 0; cbase < nseq; cbase += kExecChunk) {
            // ---- 2 jumping: thread t carries sequences cbase + t + 1024 k
            uint32_t F[kExecPer], MI[kExecPer];
            uint32_t act = 0;
#pragma unroll
            for (int k = 0; k < kExecPer; k++) {
                const uint32_t i = cbase + (uint32_t)k * kExecThreads + t;
                F[k] = 0, MI[k] = 0;
                if (i < nseq && jump_init(so[i], &F[k], &MI[k])) act |= 1u << k;
            }
            const uint32_t stop_below = min(nseq - cbase, kExecChunk) / kExecStopShare;
            if (t == 0) moved_cnt[0] = moved_cnt[1] = 0;
            __syncthreads();
            for (int round = 0; round < kExecMaxRounds; round++) {
                uint32_t chg = 0, nmoved = 0;
#pragma unroll
                for (int k = 0; k < kExecPer; k++) {
                    if (!((act >> k) & 1)) continue;
                    const int r = jump_look(pend, start, out, &F[k], &MI[k], so + cbase + (uint32_t)k * kExecThreads + t);
                    if (r == kJumpStop) {
                        act &= ~(1u << k);
                        continue;
                    }
                    nmoved++;
                    if (r == kJumpPublish) chg |= 1u << k;
                    else chg |= 1u << 16;  // (moved, nothing to publish)
                }
                nmoved = __reduce_add_sync(0xFFFFFFFFu, nmoved);
                if ((t & 31) == 0 && nmoved) atomicAdd(&moved_cnt[round & 1], nmoved);
                __syncthreads();  // every offset has been read
#pragma unroll
                for (int k = 0; k < kExecPer; k++)
                    if ((chg >> k) & 1) jump_publish(out, F[k], MI[k]);
                if (t == 0) moved_cnt[(round + 1) & 1] = 0;
                if (!__syncthreads_or((int)chg)) break;
                if (moved_cnt[round & 1] < stop_below) break;  // (uniform: read by everyone between the same two barriers)
            }
            // ---- 3 copies: in order per thread; a warp polls until its 32 current matches are copied
#pragma unroll
            for (int k = 0; k < kExecPer; k++) {
                const uint32_t i = cbase + (uint32_t)k * kExecThreads + t;
                CopyJob job = copy_job(i < nseq ? so[i] : 0, F[k], MI[k]);
                bool waiting = job.ml != 0;
                // (the spin bound is insurance, not logic: dependencies point backwards, so the earliest pending match is always
                // ready and every poll loop ends; should that reasoning ever be wrong, the frame goes back to the host instead
                // of hanging the GPU)
                for (uint32_t spins = 0; __any_sync(0xFFFFFFFFu, waiting); spins++) {
                    if (waiting && copy_ready(pend, job)) {
                        __threadfence_block();  // the bytes behind the cleared bits
                        copy_match(out, job);
                        __threadfence_block();
                        pend_clear(pend, job.m, job.ml);
                        waiting = false;
                    }
                    if (spins >= kExecMaxSpins) {
                        *bad = 1;
                        waiting = false;
                    }
                }
            }
            __syncthreads();
            if (*bad) return zd::kZdFallback;
        }
        pos += (uint32_t)total_out;
    }
    if (pos != cap) return zd::kZdFallback;
    {
        const uint4 *s4 = (const uint4 *)out;
        uint4 *d4 = (uint4 *)dst;
        const uint32_t n16 = (cap + 15) / 16;
        for (uint32_t k = t; k < n16; k += kExecThreads) d4[k] = s4[k];
    }
    return zd::kZdOk;
}

}  // namespace zd3
}  // namespace fheb
