// seq_host.cpp — host harness for the per-lane logic of the throughput path
// (claxon_b200/csrc/clx_lanes.h).  Test infrastructure only (tests/test_seq_host.py): it runs the very
// code the CUDA kernels run per lane — IndexLane once per frame, SubLane once per subframe, in the same
// head / groups-of-eight / tail order as decode_subframes_kernel — with plain loads instead of the
// shared-memory ring, then applies a scalar restatement of the kernel's prediction arithmetic so the
// result can be compared with known PCM.  Build: g++ -O2 -shared -fPIC -Iinclude.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../claxon_b200/csrc/clx_lanes.h"

namespace {

struct HostIO {
    const uint8_t* base = nullptr;  // frame's 16-byte aligned base
    uint64_t avail = 0;             // bytes readable from base
    uint32_t word(uint32_t wi) const {
        uint8_t b[4] = {0, 0, 0, 0};
        for (int i = 0; i < 4; i++) {
            const uint64_t p = (uint64_t)wi * 4 + i;
            if (p < avail) b[i] = base[p];
        }
        return ((uint32_t)b[0] << 24) | ((uint32_t)b[1] << 16) | ((uint32_t)b[2] << 8) | b[3];
    }
    uint32_t wnext = 0;
    void seek_next(uint32_t wi) { wnext = wi; }
    uint32_t next_raw() { return __builtin_bswap32(word(wnext++)); }
    void ensure(uint32_t) {}
    void ensure_near(uint32_t) {}
    bool prefetch_group(uint32_t) { return true; }
    void prefetch_run(uint32_t, uint32_t) {}
};

// The index lane's walk as index_frames_kernel schedules it: runs of up to `run_groups` (<= IndexLane::RUN) groups,
// fewer at a partition's end, slow steps for everything else.  stats (optional): [0] runs of run_groups groups,
// [1] shorter runs, [2 + j] runs that ended at their group j on a code that did not fit the window (j < 8).
// False: run-away.
bool walk_index(clx::IndexLane<HostIO>& I, uint32_t run_groups, uint64_t* stats) {
    uint64_t guard = 0;
    while (!I.done()) {
        if (I.fast_ready()) {
            const uint32_t g = I.rc.n_fast < run_groups ? I.rc.n_fast : run_groups;
            const uint32_t n0 = I.rc.n_left;
            I.run(run_groups);
            if (stats) {
                stats[g == run_groups ? 0 : 1]++;
                if (I.mode == clx::SEQ_RUN && !I.rc.wvalid) {  // the run ended early (still in its partition)
                    const uint32_t done = (n0 - I.rc.n_left) / 8;
                    if (done < 8) stats[2 + done]++;
                }
            }
        } else {
            I.slow_step();
        }
        if (++guard > (1ull << 32)) return false;
    }
    return true;
}

}  // namespace

// The index lane alone, with runs of `run_groups` groups: per subframe slot (n * CH of them, CH = the channel count
// rounded up to a power of two) the bit at which its residual starts, 0xffffffff for slots the frame does not
// use; per frame 0 (walked) or -2 (declined).  stats as walk_index.  Returns CH, or -1 on a run-away.
extern "C" int seq_host_index(const uint8_t* bytes, uint64_t nbytes, const clx_frame_desc* descs, uint32_t n,
                              uint32_t run_groups, uint32_t* res_bit, int32_t* status, uint64_t* stats) {
    uint32_t max_ch = 1;
    for (uint32_t i = 0; i < n; i++)
        if (descs[i].n_channels > max_ch) max_ch = descs[i].n_channels;
    uint32_t CH = 1;
    while (CH < max_ch) CH <<= 1;
    std::vector<clx::SeqParams> params(CH);
    for (uint32_t f = 0; f < n; f++) {
        const clx_frame_desc& d = descs[f];
        const uint64_t aligned = d.byte_offset & ~15ull;
        clx::IndexLane<HostIO> I;
        I.rc.io.base = bytes + aligned;
        I.rc.io.avail = nbytes - aligned;
        for (auto& p : params) p.res_bit = 0xffffffffu;
        I.init(d, params.data(), CH);
        if (!walk_index(I, run_groups, stats)) return -1;
        status[f] = I.ok() ? 0 : -2;
        for (uint32_t c = 0; c < CH; c++) res_bit[(size_t)f * CH + c] = c < d.n_channels ? params[c].res_bit : 0xffffffffu;
    }
    return (int)CH;
}

// head_pad: extra groups of eight samples taken one by one before the grouped part starts, as happens
// to a lane whose warp holds a subframe of a higher order; odd values also make the speculative group take one
// code per window refill throughout (as in a warp where some lane's Rice parameter is above PAIR_KMAX).  stats[0] += fast groups, stats[1] += slow codes.
extern "C" int seq_host_decode(const uint8_t* bytes, uint64_t nbytes, const clx_frame_desc* descs, uint32_t n,
                               uint32_t head_pad, int32_t* out, clx_frame_result* results, uint64_t* stats) {
    uint32_t max_ch = 1;
    for (uint32_t i = 0; i < n; i++)
        if (descs[i].n_channels > max_ch) max_ch = descs[i].n_channels;
    uint32_t CH = 1;
    while (CH < max_ch) CH <<= 1;
    std::vector<clx::SeqParams> params((size_t)n * CH);
    memset(params.data(), 0xCD, params.size() * sizeof(clx::SeqParams));
    for (uint32_t f = 0; f < n; f++) {
        const clx_frame_desc& d = descs[f];
        const uint64_t aligned = d.byte_offset & ~15ull;
        results[f].status = -2;
        results[f].consumed = 0;
        // ---- index lane ----
        clx::IndexLane<HostIO> I;
        I.rc.io.base = bytes + aligned;
        I.rc.io.avail = nbytes - aligned;
        I.init(d, params.data() + (size_t)f * CH, CH);
        if (!walk_index(I, clx::IndexLane<HostIO>::RUN, nullptr)) return -1;  // run-away
        if (!I.ok()) continue;
        // ---- one subframe lane per channel ----
        const uint32_t bs = d.block_size;
        const uint32_t bit0 = (uint32_t)(d.byte_offset & 15) * 8;
        int32_t* fo = out + d.out_offset;
        bool ok = true;
        for (uint32_t c = 0; c < d.n_channels && ok; c++) {
            const clx::SeqParams& sp = params[(size_t)f * CH + c];
            clx::SubLane<HostIO> L;
            L.rc.io.base = bytes + aligned;
            L.rc.io.avail = nbytes - aligned;
            L.init(sp, bs, bit0 + d.byte_len * 8);
            const uint32_t order = (uint32_t)sp.order;
            uint32_t head_end = ((order + 7u) & ~7u) + 8u * head_pad;
            if (head_end > bs) head_end = bs;
            const uint32_t bulk_end = head_end + ((bs - head_end) & ~7u);
            int32_t* s = fo + (size_t)c * bs;
            auto predict = [&](uint32_t t, int32_t r) {
                long long acc = 0;
                for (uint32_t j = 0; j < order; j++) acc += (long long)sp.coefs[j] * (long long)s[t - 1 - j];
                s[t] = (int32_t)((uint32_t)(int32_t)(acc >> sp.shift) + (uint32_t)r);
            };
            auto guarded = [&](uint32_t t0, uint32_t t1) {
                for (uint32_t t = t0; t < t1; t++) {
                    if (t < order) { s[t] = sp.warm[t]; continue; }
                    const int32_t r = L.next();
                    if (stats) stats[1]++;
                    predict(t, r);
                }
            };
            guarded(0, head_end);
            if (bulk_end > head_end) {
                // the kernel's software pipeline: a trip consumes the residuals the previous trip produced and
                // produces the next group speculatively (spec_group), falling back to the ordinary route
                int32_t ra[8], rb[8];
                auto produce = [&](int32_t (&dst)[8], bool try_fast) {
                    bool got = false;
                    if (try_fast) {
                        if (!L.fast()) L.prepare();
                        if (L.fast()) got = L.fast_group(dst);
                    }
                    if (got) { if (stats) stats[0]++; }
                    else {
                        for (int i = 0; i < 8; i++) dst[i] = L.next();
                        if (stats) stats[1] += 8;
                    }
                };
                auto consume = [&](const int32_t (&r)[8], uint32_t t) {
                    for (uint32_t i = 0; i < 8; i++) predict(t + i, r[i]);
                };
                auto step = [&](const int32_t (&cons)[8], int32_t (&prod)[8], uint32_t t) {
                    // the warp takes the smallest number of codes per refill any of its lanes allows: emulate
                    // neighbours with larger Rice parameters through head_pad
                    if (!L.fast()) L.quick_prepare();
                    uint32_t nc = L.spec_cap();
                    if ((head_pad & 1u) && nc > 1) nc >>= 1;
                    const bool good = nc == 2 ? L.spec_group<2>(prod) : L.spec_group<1>(prod);
                    consume(cons, t);
                    if (good) { if (stats) stats[0]++; }
                    else produce(prod, true);
                };
                produce(ra, true);
                uint32_t t = head_end;
                while (t + 16 < bulk_end) {
                    step(ra, rb, t);
                    step(rb, ra, t + 8);
                    t += 16;
                }
                if (t + 8 < bulk_end) {
                    step(ra, rb, t);
                    t += 8;
                    consume(rb, t);
                } else consume(ra, t);
            }
            guarded(bulk_end, bs);
            const uint32_t end_bit = L.finish();
            if (!L.ok()) { ok = false; break; }
            if (c + 1 == d.n_channels) {
                const uint32_t consumed = ((end_bit - bit0 + 7) >> 3) + 2;
                if (consumed > d.byte_len) { ok = false; break; }
                results[f].consumed = consumed;
            }
            for (uint32_t t = 0; t < bs; t++) s[t] = (int32_t)((uint32_t)s[t] << sp.wasted);
        }
        if (!ok) continue;
        results[f].status = 0;
        // decorrelation (src/frame.rs:319-389)
        if (d.channel_assignment >= 8) {
            int32_t *a = fo, *b = fo + bs;
            for (uint32_t t = 0; t < bs; t++) {
                const uint32_t x = (uint32_t)a[t], y = (uint32_t)b[t];
                if (d.channel_assignment == 8) b[t] = (int32_t)(x - y);
                else if (d.channel_assignment == 9) a[t] = (int32_t)(x + y);
                else {
                    const uint32_t m = (x << 1) | (y & 1u);
                    a[t] = ((int32_t)(m + y)) >> 1;
                    b[t] = ((int32_t)(m - y)) >> 1;
                }
            }
        }
    }
    return 0;
}
