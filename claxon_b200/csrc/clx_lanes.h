// clx_lanes.h — the per-lane halves of the throughput path (clx_fused.cu).
//
// FLAC gives no subframe lengths: channel n+1 starts at the bit where channel n ended (reference
// src/frame.rs:702-742), so something has to walk channel n before channel n+1 can be touched.  The
// throughput path splits that into two lane programs:
//
//   IndexLane — ONE LANE PER FRAME.  Parses every subframe header, the warm-up samples and the
//       predictor parameters (src/subframe.rs:29-91, :382-415, :651-701) and records them per subframe
//       together with the bit position at which the subframe's residual starts.  The residuals of all
//       channels but the last are only SKIPPED (unary run + k bits per code, src/subframe.rs:336-348):
//       no value is formed, nothing is stored.
//   SubLane  — ONE LANE PER SUBFRAME.  Starts at the recorded bit, decodes the Rice partitions
//       (src/subframe.rs:236-380) eight codes per trip and hands the residuals, in registers, to the
//       recurrence of the same lane (predict_fixed / predict_lpc_*, src/subframe.rs:417-474, :524-614).
//
// No residual ever goes through memory.  The logic lives in this header, free of CUDA built-ins, so
// that the very same code runs on the host inside the test harness (tools/seq_host.cpp, driven by
// tests/test_seq_host.py).  All memory traffic goes through the `IO` policy: on the device a
// shared-memory ring fed from global memory, on the host plain loads.
//
// Anything irregular (malformed input of any kind, the Rice escape code) is not guessed at: the frame
// is flagged and the generic kernel (clx_decode.cu), which owns claxon's error precedence, decodes it.
#ifndef CLX_LANES_H
#define CLX_LANES_H
#include <stdint.h>

#include "claxon_b200.h"

#ifdef __CUDACC__
#define CLX_HD __host__ __device__ __forceinline__
#else
#define CLX_HD inline
#endif

namespace clx {

enum : int32_t { SUB_PREDICTED = 0, SUB_VERBATIM = 1, SUB_CONSTANT = 2 };

// One per subframe; written by the index lane, read by the subframe lane.
struct SeqParams {
    int32_t order;      // predictor order; 0 = the residual is the sample (verbatim / fixed-0)
    int32_t shift;      // qlp shift (0 for fixed predictors)
    int32_t wasted;     // wasted bits per sample (src/subframe.rs:216-225)
    uint32_t absum;     // sum |coef|
    uint32_t res_bit;   // bit position, from the frame's 16-byte aligned base, of: the residual header
                        // (predicted), the first sample (verbatim), the end of the subframe (constant)
    int32_t kind;       // SUB_*
    uint32_t sfbps;     // bits per sample of this subframe (frame bps + side bit - wasted)
    uint32_t reserved;
    int16_t coefs[32];  // coefs[j] multiplies s[t-1-j]
    int32_t warm[32];   // warm-up samples s[0..order)
};
static_assert(sizeof(SeqParams) == 224, "SeqParams layout");

CLX_HD uint32_t hd_clz(uint32_t v) {
#ifdef __CUDA_ARCH__
    return (uint32_t)__clz((int)v);
#else
    return v ? (uint32_t)__builtin_clz(v) : 32u;
#endif
}
CLX_HD uint32_t hd_msb(uint32_t v) {  // index of the most significant set bit; 0xffffffff for v == 0
#ifdef __CUDA_ARCH__
    uint32_t r;
    asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(v));
    return r;
#else
    return v ? 31u - (uint32_t)__builtin_clz(v) : 0xffffffffu;
#endif
}
CLX_HD uint32_t hd_neg_lsb(uint32_t u) {  // 0 - (u & 1)
#ifdef __CUDA_ARCH__
    int32_t r;
    asm("bfe.s32 %0, %1, 0, 1;" : "=r"(r) : "r"(u));
    return (uint32_t)r;
#else
    return 0u - (u & 1u);
#endif
}
// upper 32 bits of (hi:lo) << (n & 31)
CLX_HD uint32_t hd_fsl(uint32_t hi, uint32_t lo, uint32_t n) {
#ifdef __CUDA_ARCH__
    return __funnelshift_l(lo, hi, n);
#else
    n &= 31;
    return n ? (hi << n) | (lo >> (32 - n)) : hi;
#endif
}
// lower 32 bits of (hi:lo) >> (n & 31)
CLX_HD uint32_t hd_fsr(uint32_t hi, uint32_t lo, uint32_t n) {
#ifdef __CUDA_ARCH__
    return __funnelshift_r(lo, hi, n);
#else
    n &= 31;
    return n ? (lo >> n) | (hi << (32 - n)) : lo;
#endif
}
CLX_HD uint32_t hd_bswap(uint32_t v) {
#ifdef __CUDA_ARCH__
    return __byte_perm(v, 0, 0x0123);
#else
    return __builtin_bswap32(v);
#endif
}
CLX_HD int32_t hd_sext(uint32_t v, uint32_t bits) {  // bits in [1, 32]
    return ((int32_t)(v << (32 - bits))) >> (32 - bits);
}

enum : uint32_t { SEQ_SUBFRAME = 0, SEQ_PART = 1, SEQ_RUN = 2, SEQ_DONE = 3 };

// IO policy (DeviceIO in clx_fused.cu, HostIO in tools/seq_host.cpp):
//   uint32_t word(uint32_t wi)            big-endian word `wi` of the frame (relative to its 16-byte aligned base)
//   void ensure(uint32_t bitpos)          the bits from bitpos on (ring size minus slack) are readable through word()
//   bool prefetch_group(uint32_t bitpos)  steady-state refill, once per fast group; false: ensure() before reading on
//   void prefetch_run(uint32_t bitpos, uint32_t quads)   steady-state refill, once per run of groups (skip_run) that
//                                         consumes at most `quads` 16-byte quads from bitpos on
//   void seek_next(uint32_t wi), uint32_t next_raw()   sequential word reads, bytes as stored (the register window's refill)
//   void ensure_near(uint32_t bitpos)     cheap: the next 16 bytes from bitpos are readable (refills, blocking, only if not)

// ---------------------------------------------------------------------------------
// Bit window + Rice partition state shared by both lanes
// ---------------------------------------------------------------------------------
// Codes of a partition are taken two per window refill when its Rice parameter is at most PAIR_KMAX, else one
// (see codes8()).  A pair needs its two codes to be at most 32 bits long together; the bound is low because a
// lane that fails takes its whole WARP through the slow branch: the per-lane failure rate has to be ~1e-4 per
// group, i.e. (two-sided geometric residuals, mean quotient ~1) quotient sums above ~18 only.
constexpr uint32_t PAIR_KMAX = 6;

template <class IO>
struct RiceCursor {
    IO io;
    uint32_t o;           // bit cursor, relative to the frame's 16-byte aligned base
    uint32_t limit;       // first bit past the frame's available bytes
    // Register window over the words at o >> 5 (valid while n_fast != 0): W0, W1 big-endian, W2 the next word
    // as loaded (little-endian).  W2 is byte-swapped only when it moves up, one refill later, so the swap never
    // waits for the shared-memory load that produced it.
    uint32_t W0, W1, W2;
    uint32_t n_left, parts_left, per, order, pbits;
    uint32_t k, Kneg, K30;
    uint32_t ncap;        // codes per window refill this partition allows: 2 or 1
    uint32_t n_fast;      // groups of eight codes the fast path may take before anything else has to happen
    bool ok, first_part;
    bool wvalid;          // W0..W2 are seated at the cursor (so single codes and partition headers can use them)

    CLX_HD void reset(uint32_t start_bit, uint32_t limit_bit) {
        o = start_bit; limit = limit_bit;
        W0 = W1 = W2 = 0;
        n_left = 0; parts_left = 0; per = 0; order = 0; pbits = 4;
        k = 0; Kneg = 0xffffffffu; K30 = 30; ncap = 1;
        n_fast = 0;
        ok = true; first_part = false; wvalid = false;
    }
    CLX_HD void fail() { ok = false; n_left = 0; parts_left = 0; n_fast = 0; wvalid = false; }
    CLX_HD uint32_t peek32(uint32_t pos) { return hd_fsl(io.word(pos >> 5), io.word((pos >> 5) + 1), pos); }
    CLX_HD uint32_t bits(uint32_t pos, uint32_t n) { return n ? peek32(pos) >> (32 - n) : 0u; }  // n <= 32
    // Seats the register window at the cursor and opens the fast path for the rest of the partition.
    CLX_HD void window_seek() {
        io.ensure_near(o);
        const uint32_t wi = o >> 5;
        W0 = io.word(wi); W1 = io.word(wi + 1);
        io.seek_next(wi + 2);
        W2 = io.next_raw();
        n_fast = n_left >> 3;
        wvalid = true;
    }
    // Moves the seated window forward by n bits (n <= 32).
    CLX_HD void window_advance(uint32_t n) {
        const uint32_t on = o + n;
        if ((on ^ o) & 32u) { W0 = W1; W1 = hd_bswap(W2); W2 = io.next_raw(); }
        o = on;
    }

    // residual header (src/subframe.rs:236-304) at the cursor; `bs` = block size, `ord` = predictor order
    CLX_HD void residual_header(uint32_t bs, uint32_t ord) {
        io.ensure(o);
        const uint32_t rh = bits(o, 6);  // 2-bit coding method, 4-bit partition order
        o += 6;
        const uint32_t method = rh >> 4, po = rh & 15u;
        if (method > 1) { fail(); return; }
        const uint32_t n_part = 1u << po;
        if ((bs & ((n_part - 1u) & 0xffffu)) != 0) { fail(); return; }
        per = bs >> po;
        order = ord;
        if (ord > per) { fail(); return; }
        pbits = method == 0 ? 4u : 5u;
        parts_left = n_part;
        first_part = true;
        n_left = 0;
        n_fast = 0;
        wvalid = false;
    }
    // partition header (src/subframe.rs:310-319, :358-367)
    CLX_HD void do_part() {
        io.ensure_near(o);
        k = bits(o, pbits);
        o += pbits;
        n_fast = 0;
        wvalid = false;
        if (k == (1u << pbits) - 1u) { fail(); return; }  // escape code: Unsupported in the reference
        set_parameter();
    }
    CLX_HD void set_parameter() {
        n_left = first_part ? per - order : per;
        first_part = false;
        parts_left--;
        const uint32_t K = 1u << k;
        K30 = (30u - k) * K;
        Kneg = 0u - K;
        ncap = k <= PAIR_KMAX ? 2u : 1u;
        if (o > limit) fail();
    }
    // The next partition's header straight from the seated window — the common way from one partition to the
    // next: no shared-memory round trip, the window stays seated and the fast path open.  Precondition: wvalid,
    // n_left == 0, parts_left != 0, not the first partition.
    CLX_HD void quick_part() {
        k = hd_fsl(W0, W1, o) >> (32u - pbits);
        window_advance(pbits);
        if (k == (1u << pbits) - 1u) { fail(); return; }
        set_parameter();
        n_fast = n_left >> 3;
    }
    // Moves to the partition that holds the next residual (empty partitions still carry a parameter,
    // src/subframe.rs:283-288).  False: nothing left, or failed.
    CLX_HD bool settle() {
        while (n_left == 0) {
            if (!ok || parts_left == 0) return false;
            do_part();
        }
        return ok;
    }
    // Called when n_fast == 0 and a group of eight is wanted: partition switch and window seat.
    CLX_HD void prepare() {
        if (!ok) return;
        if (n_left == 0 && parts_left != 0) {
            if (wvalid && !first_part) { quick_part(); if (n_left != 0 || !ok) return; }  // (an empty partition: the slow way)
            settle();
        }
        if (ok && n_left >= 8 && !wvalid) window_seek();
        else if (ok && wvalid) n_fast = n_left >> 3;
    }

    // (q << k) | r of the code whose 32-bit window is `hi` with its terminator at bit m = sh + k, then
    // rice_to_signed (src/subframe.rs:157-170): (u >> 1) ^ -(u & 1).
    CLX_HD int32_t code_value(uint32_t hi, uint32_t sh) const {
        const uint32_t v = hi >> (sh & 31u);      // K + r
        const uint32_t u = sh * Kneg + (v + K30); // (q << k) | r = (30 - k - sh) * K + v,  q = 31 - k - sh
        return (int32_t)((u >> 1) ^ hd_neg_lsb(u));
    }

    // ---- eight Rice codes (src/subframe.rs:336-348) from the register window ----
    // NC codes share one 32-bit window and one refill test: the window of the next code is the previous one's
    // shifted left by its length (zeros come in at the bottom), which is all it needs as long as the NC codes
    // TOGETHER are at most 32 bits long.  A code that does not fit — its terminator or its remainder beyond the
    // window, or no terminator at all (bfind of 0 is 0xffffffff) — makes the sum of the lengths exceed 32 (for one
    // code alone: makes sh negative), so that one comparison per refill covers everything; what was decoded after such a code is meaningless
    // (but harmless: every shared-memory address is masked into the lane's ring) and `bad` is returned.
    // NC = 1 takes any code of up to 32 bits; NC = 2 is for partitions with k <= PAIR_KMAX.
    template <int NC, bool VALUES>
    CLX_HD bool codes8(int32_t (&e)[8]) {
        bool bad = false;
#pragma unroll
        for (int i = 0; i < 8; i += NC) {
            uint32_t x = hd_fsl(W0, W1, o);
            uint32_t t = 0;  // sum of sh = m - k over the NC codes; a code is 32 - sh bits long
#pragma unroll
            for (int j = 0; j < NC; j++) {
                const uint32_t sh = hd_msb(x) - k;  // terminator at bit m = sh + k (sh < 0: it does not fit)
                if (VALUES) e[i + j] = code_value(x, sh);
                t += sh;
                if (j + 1 < NC) x = hd_fsr(x, 0u, sh);  // x << (32 - sh): the next code's window
            }
            bad = bad || (int32_t)t < 32 * (NC - 1);  // the NC codes are longer than 32 bits together
            const uint32_t on = o - t + 32u * NC;
            if ((on ^ o) & 32u) { W0 = W1; W1 = hd_bswap(W2); W2 = io.next_raw(); }
            o = on;
        }
        return bad;
    }
    // The group, by the form the partition allows; precondition n_fast != 0.  On failure the cursor is put back
    // and the fast path closed: the caller then takes the eight codes one by one.  (A quad or pair that fails
    // only because its codes are too long TOGETHER is retried one form down first.)
    CLX_HD bool fast_group(int32_t (&e)[8]) {
        if (!io.prefetch_group(o)) io.ensure(o);  // the ring had fallen behind (a dense stretch): refill it, blocking
        const uint32_t o0 = o, w0 = W0, w1 = W1, w2 = W2;
        bool bad = ncap == 2 ? codes8<2, true>(e) : codes8<1, true>(e);
        if (bad && ncap > 1) {  // once more, one code per refill: needs the window back
            o = o0; W0 = w0; W1 = w1; W2 = w2;
            io.seek_next((o0 >> 5) + 3);
            bad = codes8<1, true>(e);
        }
        if (bad) { o = o0; n_fast = 0; wvalid = false; return false; }
        n_left -= 8;
        n_fast--;
        return true;
    }
    // ---- a run of `groups` groups of eight codes, positions only (the index lane's walk) ----
    // Preconditions: the window is seated, 1 <= groups <= MAXG, groups <= n_fast (the run stays inside the
    // partition), NC <= ncap.  One ring refill covers the whole run.  Groups are committed as they go: a group that
    // does not fit — a pair longer than 32 bits together, a code longer than the window — ends the run at its first
    // code, with the fast path closed and false returned, and the caller takes it from there (the window is re-seated
    // at the cursor, so nothing is saved here and nothing is retried).  Afterwards cursor, n_left and n_fast are what
    // `groups` single-group runs would have left.
    template <int NC, uint32_t MAXG>
    CLX_HD bool skip_run(uint32_t groups) {
        // a group is at most 8 * 16 bits = 1 quad long with two codes per 32-bit window, 8 * 32 bits with one
        io.prefetch_run(o, MAXG * (NC == 2 ? 1u : 2u));
        int32_t unused[8];
        uint32_t g = 0, o0 = o;
        bool bad = false;
#pragma unroll
        for (; g < MAXG; g++) {
            o0 = o;
            bad = codes8<NC, false>(unused);
            if (bad || g + 1 == groups) break;  // one exit test per group
        }
        g += bad ? 0u : 1u;  // groups taken
        n_left -= 8u * g;
        if (bad) { o = o0; n_fast = 0; wvalid = false; return false; }
        n_fast -= groups;
        return true;
    }
    // The same group SPECULATIVELY and branch-free, whatever the lane's state (every memory access it makes is
    // safe in any state): the caller learns afterwards whether the residuals are real.  This lets the caller put
    // the group in one basic block with independent work (the previous group's prediction), so that the two
    // dependency chains — and the ALU-heavy bit scan and the multiply-add-heavy recurrence — interleave.
    // NC may be at most the `ncap` of every lane that is on the fast path.
    template <int NC>
    CLX_HD bool spec_group(int32_t (&e)[8]) {
        const bool was_fast = n_fast != 0;
        const bool ring_ok = io.prefetch_group(o);
        const uint32_t o0 = o;
        const bool bad = codes8<NC, true>(e);
        const bool good = was_fast && ring_ok && !bad;
        o = good ? o : o0;
        n_left = good ? n_left - 8 : n_left;
        n_fast = good ? n_fast - 1 : 0u;
        wvalid = good;  // a group that does not count has moved the registers but not the cursor
        return good;
    }
    // ---- one Rice code (precondition n_left > 0): from the seated window when it fits, else the long way ----
    template <bool VALUES>
    CLX_HD int32_t one_code() {
        if (!wvalid) window_seek();
        else io.ensure_near(o);
        const uint32_t x = hd_fsl(W0, W1, o);
        const uint32_t sh = hd_msb(x) - k;
        if ((int32_t)sh < 0) return slow_code();  // longer than the window
        const int32_t e = VALUES ? code_value(x, sh) : 0;
        window_advance(32u - sh);
        n_left--;
        n_fast = n_left >> 3;
        return e;
    }
    // ---- one Rice code of any shape; precondition n_left > 0 ----
    CLX_HD int32_t slow_code() {
        n_fast = 0;
        wvalid = false;
        uint32_t q = 0;
        uint32_t v;
        for (;;) {
            io.ensure(o);
            v = peek32(o);
            if (v != 0) break;
            q += 32; o += 32;
            if (o > limit) { fail(); return 0; }
        }
        const uint32_t z = hd_clz(v);
        q += z;
        o += z + 1;
        const uint32_t r = bits(o, k);
        o += k;
        n_left--;
        const uint32_t u = (q << k) | r;  // wrapping, as the reference's u32 arithmetic
        return (int32_t)((u >> 1) ^ (0u - (u & 1u)));
    }
};

// ---------------------------------------------------------------------------------
// Index lane: one per frame
// ---------------------------------------------------------------------------------
template <class IO>
struct IndexLane {
    RiceCursor<IO> rc;
    SeqParams* params;  // the frame's CH records
    uint32_t bs, nch, ca, fbps, bit0, byte_len;
    uint32_t mode, ch;
    uint32_t slow_budget;  // codes to take one by one after a group that did not fit the window

    CLX_HD void init(const clx_frame_desc& d, SeqParams* p, uint32_t max_channels) {
        params = p;
        bs = d.block_size; nch = d.n_channels; ca = d.channel_assignment; fbps = d.bits_per_sample;
        byte_len = d.byte_len;
        bit0 = (uint32_t)(d.byte_offset & 15) * 8;
        rc.reset(bit0 + (uint32_t)d.header_len * 8, bit0 + d.byte_len * 8);
        mode = SEQ_SUBFRAME; ch = 0; slow_budget = 0;
        if (nch > max_channels || nch == 0 || fbps == 0) fail();
    }
    CLX_HD void fail() { rc.fail(); mode = SEQ_DONE; }
    CLX_HD bool ok() const { return rc.ok; }
    CLX_HD bool done() const { return mode == SEQ_DONE; }
    static constexpr uint32_t RUN = 4;  // at most this many groups of eight codes per run
    // slow_budget of a lane whose group of pairs did not fit: its next slow step retries the group one code per
    // window refill before it takes the codes one by one
    static constexpr uint32_t RETRY_SINGLES = 9;
    CLX_HD bool fast_ready() const { return mode == SEQ_RUN && rc.n_fast != 0; }
    // A run of min(n_fast, cap) groups of eight codes (cap <= RUN), two codes per window refill where the
    // partition's Rice parameter allows; then the next partition if this one has ended.  A partition's last groups
    // are a shorter run, so that a warp whose lanes cross partition boundaries at different times stays in its
    // tight loop.
    CLX_HD void run(uint32_t cap = RUN) {
        const uint32_t groups = rc.n_fast < cap ? rc.n_fast : cap;
        const bool good = rc.ncap == 2 ? rc.template skip_run<2, RUN>(groups) : rc.template skip_run<1, RUN>(groups);
        slow_budget = good ? slow_budget : rc.ncap == 2 ? RETRY_SINGLES : 8u;
        if (good) after_group();
    }
    CLX_HD void after_group() {
        if (rc.n_left == 0) {
            if (rc.parts_left == 0) end_of_body();
            else if (rc.wvalid) {
                // The next partition's parameter straight from the seated window, so that a warp whose lanes cross
                // partition boundaries all the time (partitions of 32 codes: every fourth group) stays in its tight loop.
                rc.quick_part();
                if (!rc.ok) fail();
            }
        }
    }
    CLX_HD void end_of_body() {
        if (rc.o > rc.limit) { fail(); return; }
        ch++;
        mode = SEQ_SUBFRAME;
    }

    // subframe header, warm-up, predictor parameters; then either stop (last channel) or start skipping
    CLX_HD void do_subframe() {
        IO& io = rc.io;
        uint32_t& o = rc.o;
        io.ensure(o);
        uint32_t bps = fbps;
        if (ca == 9) bps += (ch == 0);                   // side/right: side first (src/frame.rs:725)
        else if (ca == 8 || ca == 10) bps += (ch == 1);  // src/frame.rs:717, :736
        SeqParams* sp = params + ch;
        const bool last = ch + 1 == nch;
        // subframe header (src/subframe.rs:29-91)
        const uint32_t head = rc.bits(o, 8);
        o += 8;
        if (head & 0x80u) { fail(); return; }
        const uint32_t code = (head >> 1) & 0x3fu;
        uint32_t order = 0;
        int type;
        if (code == 0) type = 0;
        else if (code == 1) type = 1;
        else if ((code & 0x3eu) == 0x02u || (code & 0x3cu) == 0x04u || (code & 0x30u) == 0x10u) { fail(); return; }
        else if ((code & 0x38u) == 0x08u) { order = code & 7u; if (order > 4) { fail(); return; } type = 2; }
        else { order = (code & 0x1fu) + 1; type = 3; }
        uint32_t wasted = 0;
        if (head & 1u) {
            const uint32_t v = rc.peek32(o);
            if (v == 0) { fail(); return; }  // > 31 wasted bits: an error for the generic kernel to name
            const uint32_t q = hd_clz(v);
            wasted = q + 1;
            o += q + 1;
        }
        if (wasted >= bps) { fail(); return; }
        const uint32_t sfbps = bps - wasted;
        if (sfbps > 32) { fail(); return; }
        if ((type == 2 || type == 3) && order > bs) { fail(); return; }
        sp->wasted = (int32_t)wasted;
        sp->sfbps = sfbps;
        sp->reserved = 0;
        if (type == 0) {  // constant (src/subframe.rs:382-394): an order-1 predictor with coefficient 1 over zero residuals
            const int32_t v = hd_sext(rc.bits(o, sfbps), sfbps);
            o += sfbps;
            sp->kind = SUB_CONSTANT;
            sp->order = 1; sp->shift = 0; sp->absum = 1; sp->coefs[0] = 1; sp->warm[0] = v;
            sp->res_bit = o;
            if (o > rc.limit) { fail(); return; }
            if (last) { mode = SEQ_DONE; return; }
            ch++;
            return;  // mode stays SEQ_SUBFRAME
        }
        if (type == 1) {  // verbatim (src/subframe.rs:397-415): the samples are the residuals of an order-0 predictor
            sp->kind = SUB_VERBATIM;
            sp->order = 0; sp->shift = 0; sp->absum = 0;
            sp->res_bit = o;
            if (last) { mode = SEQ_DONE; return; }
            const uint64_t end = (uint64_t)o + (uint64_t)bs * sfbps;
            if (end > rc.limit) { fail(); return; }
            o = (uint32_t)end;
            ch++;
            return;
        }
        for (uint32_t i = 0; i < order; i++) {  // warm-up
            if ((i & 3u) == 0) io.ensure(o);
            sp->warm[i] = hd_sext(rc.bits(o, sfbps), sfbps);
            o += sfbps;
        }
        if (o > rc.limit) { fail(); return; }
        io.ensure(o);
        uint32_t shift = 0, absum = 0;
        if (type == 3) {  // src/subframe.rs:669-701
            const uint32_t pq = rc.bits(o, 9);  // 4-bit precision-1, 5-bit signed shift
            o += 9;
            const uint32_t prec_m1 = pq >> 5;
            if (prec_m1 == 15) { fail(); return; }
            const uint32_t precision = prec_m1 + 1;
            const int32_t sh = hd_sext(pq & 31u, 5);
            if (sh < 0) { fail(); return; }
            shift = (uint32_t)sh;
            for (uint32_t j = 0; j < order; j++) {
                if ((j & 7u) == 0) io.ensure(o);
                const int32_t c = hd_sext(rc.bits(o, precision), precision);
                o += precision;
                sp->coefs[j] = (int16_t)c;
                absum += (uint32_t)(c < 0 ? -c : c);
            }
        } else {  // rows of src/subframe.rs:427-431; coefs[0] multiplies s[t-1]
            const uint32_t packed = order == 1 ? 0x00000001u : order == 2 ? 0x0000ff02u
                                  : order == 3 ? 0x0001fd03u : order == 4 ? 0xff04fa04u : 0u;
            for (uint32_t j = 0; j < order; j++) {
                const int32_t c = (int32_t)(int8_t)(packed >> (8 * j));
                sp->coefs[j] = (int16_t)c;
                absum += (uint32_t)(c < 0 ? -c : c);
            }
        }
        sp->kind = SUB_PREDICTED;
        sp->order = (int32_t)order; sp->shift = (int32_t)shift; sp->absum = absum;
        sp->res_bit = o;
        if (o > rc.limit) { fail(); return; }
        if (last) { mode = SEQ_DONE; return; }
        rc.residual_header(bs, order);
        if (!rc.ok) { fail(); return; }
        mode = SEQ_RUN;
        if (!rc.settle()) {  // no residual at all (order == block size, every partition empty)
            if (!rc.ok) { fail(); return; }
            end_of_body();
            return;
        }
        if (rc.n_left >= 8) rc.window_seek();
    }

    // everything that is not a fast group
    CLX_HD void slow_step() {
        if (mode == SEQ_SUBFRAME) { do_subframe(); return; }
        if (mode != SEQ_RUN) return;
        if (rc.n_left == 0) {  // next partition (or the end of the subframe's residual)
            if (rc.parts_left != 0 && rc.wvalid && !rc.first_part) rc.quick_part();
            if (rc.ok && rc.n_left == 0 && !rc.settle()) {
                if (!rc.ok) { fail(); return; }
                end_of_body();
                return;
            }
            if (!rc.ok) { fail(); return; }
            if (rc.n_fast != 0 && slow_budget == 0) return;  // next step: a fast group
        }
        if (slow_budget == RETRY_SINGLES) {  // (n_left >= 8: the group that failed is still ahead)
            rc.window_seek();
            if (rc.template skip_run<1, 1>(1)) { slow_budget = 0; after_group(); return; }
            slow_budget = 8;  // a code longer than the window: one by one
        }
        if (slow_budget == 0 && rc.n_left >= 8) {
            if (!rc.wvalid) rc.window_seek();
            else rc.n_fast = rc.n_left >> 3;
            return;  // next step: a fast group
        }
        rc.template one_code<false>();  // the last few codes of a partition, or a stretch after a group that failed
        if (slow_budget) slow_budget--;
        if (!rc.ok) { fail(); return; }
        if (rc.n_left == 0 && rc.parts_left == 0) end_of_body();
    }
};

// ---------------------------------------------------------------------------------
// Subframe lane: one per (frame, channel)
// ---------------------------------------------------------------------------------
template <class IO>
struct SubLane {
    RiceCursor<IO> rc;
    uint32_t kind, sfbps;

    // `limit`: first bit past the frame's bytes; the cursor starts at sp.res_bit
    CLX_HD void init(const SeqParams& sp, uint32_t bs, uint32_t limit) {
        rc.reset(sp.res_bit, limit);
        kind = (uint32_t)sp.kind;
        sfbps = sp.sfbps;
        if (kind == SUB_PREDICTED) rc.residual_header(bs, (uint32_t)sp.order);
    }
    CLX_HD void init_idle() {
        rc.reset(0, 0);
        kind = SUB_CONSTANT; sfbps = 1;
    }
    CLX_HD bool ok() const { return rc.ok; }
    // A group of eight residuals: `if (!fast()) prepare(); if (fast()) got = fast_group(e); if (!got) eight next()`.
    CLX_HD bool fast() const { return rc.n_fast != 0; }
    CLX_HD void prepare() { if (kind == SUB_PREDICTED) rc.prepare(); }
    // The cheap part of prepare(), for the top of a trip: the next partition's header from the seated window.
    CLX_HD void quick_prepare() {
        if (kind == SUB_PREDICTED && rc.ok && rc.wvalid && rc.n_left == 0 && rc.parts_left != 0 && !rc.first_part) rc.quick_part();
    }
    CLX_HD bool fast_group(int32_t (&e)[8]) { return rc.fast_group(e); }
    // codes per refill spec_group may use for this lane (a lane off the fast path does not care)
    CLX_HD uint32_t spec_cap() const { return rc.n_fast == 0 ? 2u : rc.ncap; }
    // the same for the rest of the subframe, once its last partition has begun (parts_left == 0)
    CLX_HD uint32_t last_cap() const { return kind == SUB_PREDICTED && rc.ok ? rc.ncap : 2u; }
    template <int NC>
    CLX_HD bool spec_group(int32_t (&e)[8]) { return rc.template spec_group<NC>(e); }
    // one residual through the slow path, whatever the subframe's kind; 0 once the lane has failed
    CLX_HD int32_t next() {
        if (kind == SUB_CONSTANT || !rc.ok) return 0;
        if (kind == SUB_VERBATIM) {
            rc.io.ensure(rc.o);
            const int32_t v = hd_sext(rc.bits(rc.o, sfbps), sfbps);
            rc.o += sfbps;
            if (rc.o > rc.limit) { rc.fail(); return 0; }
            return v;
        }
        if (rc.n_left == 0) {
            if (rc.parts_left != 0 && rc.wvalid && !rc.first_part) rc.quick_part();
            if (rc.ok && rc.n_left == 0 && !rc.settle()) { rc.fail(); return 0; }  // more residuals asked for than the partitions hold
            if (!rc.ok) return 0;
        }
        return rc.template one_code<true>();
    }
    // After the last residual: the subframe must end inside the frame.  Returns the end bit.
    CLX_HD uint32_t finish() {
        if (kind == SUB_PREDICTED && rc.ok) {
            // trailing empty partitions (order == per, partition order 0) still carry their parameter
            while (rc.ok && rc.n_left == 0 && rc.parts_left != 0) rc.do_part();
            if (rc.n_left != 0 || rc.parts_left != 0) rc.fail();
        }
        if (rc.o > rc.limit) rc.fail();
        return rc.o;
    }
};

}  // namespace clx
#endif
