// plan_codec_jobs (csrc/codec_stage.h), the one job layout of the device codec's staging: payload jobs first, frames behind them
// with their pads, within the staging every caller allocates, and one layout per pair of routes for the single-call graphs.
// Built with g++ alone by tests/test_codec_stage.py; prints "ok".
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>

#include "codec_stage.h"

using namespace fheb;

#define CHECK(c)                                                       \
    do {                                                               \
        if (!(c)) {                                                    \
            std::printf("FAIL %s:%d: %s\n", __FILE__, __LINE__, #c);   \
            std::exit(1);                                              \
        }                                                              \
    } while (0)

constexpr size_t kMaxFrame = kFrameSlotBytes - 2 * kFramePad;  // the largest frame a caller accepts

struct Planned {
    std::vector<CodecJob> jobs;
    std::vector<int32_t> job;
    StagePlan plan;
};

// plans `ops` and checks every invariant the callers rely on
Planned plan_and_check(const std::vector<StageOperand> &ops) {
    Planned r;
    r.jobs.assign(ops.size(), CodecJob{});
    r.job.assign(ops.size(), -2);
    r.plan = plan_codec_jobs(ops.data(), ops.size(), r.jobs.data(), r.job.data());
    const StagePlan &p = r.plan;
    size_t lib = 0, accepted = 0;
    for (const StageOperand &o : ops) {
        lib += o.route == Route::Zstd;
        accepted += o.route == Route::Blob || o.route == Route::Zstd || o.route == Route::Packed;
    }
    const bool dev = device_inflates(lib);
    CHECK(p.jobs == (int)accepted && p.payloads <= p.jobs);
    // payload jobs are exactly [0, P)
    for (int j = 0; j < p.jobs; j++) CHECK((r.jobs[(size_t)j].kind == kJobPayload) == (j < p.payloads));
    // each accepted operand has its own job, with its destination and the kind its route and the inflate rule give
    std::vector<int> seen((size_t)p.jobs, 0);
    bool any_zstd = false, any_packed = false;
    for (size_t i = 0; i < ops.size(); i++) {
        const StageOperand &o = ops[i];
        if (o.route == Route::Reject || o.route == Route::Host) {
            CHECK(r.job[i] == -1);
            continue;
        }
        CHECK(r.job[i] >= 0 && r.job[i] < p.jobs && seen[(size_t)r.job[i]]++ == 0);
        const CodecJob &jb = r.jobs[(size_t)r.job[i]];
        CHECK(jb.slot == o.slot && jb.operand == o.operand);
        const int32_t want = o.route == Route::Packed ? kJobPacked : (o.route == Route::Zstd && dev) ? kJobZstd : kJobPayload;
        CHECK(jb.kind == want);
        any_zstd |= want == kJobZstd, any_packed |= want == kJobPacked;
        if (want != kJobPayload) CHECK(jb.src_len == o.frame_len);
    }
    CHECK(p.any_zstd == any_zstd && p.any_packed == any_packed);
    // frames: 16-byte aligned, kFramePad readable bytes on either side, padded ranges disjoint and inside [0, frame_bytes)
    size_t end = 0;
    for (int j = p.payloads; j < p.jobs; j++) {
        const CodecJob &jb = r.jobs[(size_t)j];
        CHECK(jb.src_off % 16 == 0 && jb.src_off >= kFramePad);
        CHECK(jb.src_off - kFramePad >= end);  // frame jobs are laid out in job order
        end = jb.src_off + jb.src_len + kFramePad;
        CHECK(end <= p.frame_bytes);
    }
    if (p.payloads == p.jobs) CHECK(p.frame_bytes == 0);
    return r;
}

int main() {
    CHECK(!device_inflates(kDeviceZstdMinFrames - 1) && device_inflates(kDeviceZstdMinFrames));
    CHECK(!device_inflates(127) && device_inflates(128));

    // the inflate rule through the plan: 127 libzstd frames are all inflated on the host, 128 all on the device
    for (size_t n : {size_t(127), size_t(128)}) {
        std::vector<StageOperand> ops;
        for (size_t i = 0; i < n; i++) ops.push_back(StageOperand{Route::Zstd, 60000 + i, (int32_t)i, 0});
        const Planned r = plan_and_check(ops);
        CHECK(r.plan.payloads == (n == 127 ? 127 : 0) && r.plan.any_zstd == (n == 128));
    }

    // worst-case frames fill the staging callers allocate and no more: a lane of `cap` calls stages 2 * cap frame slots,
    // an upload chunk kXferChunk (256) of them
    for (size_t m : {size_t(1), size_t(2), size_t(32), size_t(256), size_t(2048)}) {
        for (Route r : {Route::Zstd, Route::Packed}) {
            std::vector<StageOperand> ops;
            for (size_t i = 0; i < m; i++)
                ops.push_back(StageOperand{i % 2 ? r : Route::Zstd, r == Route::Packed && i % 2 ? kPackedFrameBytes : kMaxFrame,
                                           (int32_t)(i / 2), (int32_t)(i % 2)});
            const Planned p = plan_and_check(ops);
            CHECK(p.plan.frame_bytes <= m * kFrameSlotBytes);
        }
    }

    // random mixes of every route, lengths and destinations
    std::mt19937_64 rng(12345);
    for (int trial = 0; trial < 2000; trial++) {
        const size_t n = rng() % 300;
        const int zstd_bias = (int)(rng() % 4);  // some trials cross the inflate threshold
        std::vector<StageOperand> ops;
        for (size_t i = 0; i < n; i++) {
            const int pick = (int)(rng() % 8);
            Route r = pick < zstd_bias + 3 ? Route::Zstd : (Route)(rng() % 5);
            const size_t len = r == Route::Packed ? kPackedFrameBytes : 1 + rng() % kMaxFrame;
            ops.push_back(StageOperand{r, len, (int32_t)(i / 2), (int32_t)(i % 2)});
        }
        const Planned p = plan_and_check(ops);
        CHECK(p.plan.frame_bytes <= n * kFrameSlotBytes);
    }

    // a single call: one or two operands, each Zstd or Packed.  Its graph is keyed on the routes, so the jobs' offsets and
    // kinds, P and the frame bytes must not depend on the lengths of the libzstd frames (inflated on the host)
    const Route rs[2] = {Route::Zstd, Route::Packed};
    int combos = 0;
    for (int nct = 1; nct <= 2; nct++)
        for (int a = 0; a < 2; a++)
            for (int b = 0; b < (nct == 2 ? 2 : 1); b++) {
                combos++;
                Planned first;
                for (size_t len : {size_t(1), size_t(88000), size_t(100003), kMaxFrame}) {
                    std::vector<StageOperand> ops;
                    for (int k = 0; k < nct; k++) {
                        const Route r = rs[k == 0 ? a : b];
                        ops.push_back(StageOperand{r, r == Route::Packed ? kPackedFrameBytes : len, 0, k});
                    }
                    const Planned p = plan_and_check(ops);
                    CHECK(!p.plan.any_zstd && p.plan.frame_bytes <= 2 * kFrameSlotBytes);
                    if (first.jobs.empty()) {
                        first = p;
                        continue;
                    }
                    CHECK(p.plan.jobs == first.plan.jobs && p.plan.payloads == first.plan.payloads &&
                          p.plan.frame_bytes == first.plan.frame_bytes && p.plan.any_packed == first.plan.any_packed);
                    for (size_t j = 0; j < p.jobs.size(); j++) {
                        const CodecJob &x = p.jobs[j], &y = first.jobs[j];
                        CHECK(x.src_off == y.src_off && x.kind == y.kind && x.slot == y.slot && x.operand == y.operand);
                    }
                    CHECK(p.job == first.job);
                }
            }
    CHECK(combos == 6);
    std::printf("ok\n");
    return 0;
}
