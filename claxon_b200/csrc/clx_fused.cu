// clx_fused.cu — the throughput path of claxon_b200: an index pass (one lane per frame) and a fused
// entropy-decode + prediction pass (one lane per subframe).  No residual ever touches memory.
//
//   1. `index_frames_kernel` — ONE LANE PER FRAME, 32 frames per warp (clx_lanes.h: IndexLane).  FLAC
//      carries no subframe lengths (reference src/frame.rs:702-742: channel n+1 starts where channel n
//      ended), so one lane walks the frame once: subframe headers, warm-up samples and predictor
//      parameters (src/subframe.rs:29-91, :382-415, :651-701) are parsed and recorded per subframe
//      together with the bit at which its residual starts; the Rice codes of every channel but the last
//      are only stepped over (src/subframe.rs:336-348: unary run + k bits), in runs of four groups of eight
//      behind one ring refill.
//   2. `decode_subframes_kernel` — ONE LANE PER SUBFRAME.  The lane starts at the recorded bit, decodes
//      its Rice partitions eight codes per trip from a three-word register window over a per-lane
//      shared-memory ring (src/subframe.rs:236-380) and feeds the residuals, still in registers, to the
//      recurrence it runs itself: predict_fixed / predict_lpc_* (src/subframe.rs:417-474, :524-614) are
//      strictly serial (the floor in `>> qlp_shift` makes them non-associative), so the parallel axis is
//      the set of subframes — coefficients and history register-resident, eight samples per trip.
//      Samples leave through a swizzled 32x32 shared-memory transpose; the flush handles the two channels
//      of a frame together, which turns the wasted-bits shift (src/subframe.rs:216-225) and the
//      inter-channel decorrelation (src/frame.rs:319-389) into a few operations per PAIR of 16-byte
//      vectors, and writes planar i32 as whole 128-byte lines.
//
// HBM traffic per frame: its bytes once for the decode, the bytes of all channels but the last once more
// for the index pass, 224 bytes of parameters per subframe, and the planar i32 output once.
// Anything irregular is flagged (CLX_INTERNAL_NEED_GENERIC) and decoded by the generic kernel.
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "claxon_b200.h"
#include "clx_internal.h"
#include "clx_lanes.h"

namespace clx {

// ---------------------------------------------------------------------------------
// Device IO policy of a lane: a ring of RQ 16-byte quads in shared memory, fed by cp.async
// ---------------------------------------------------------------------------------
template <uint32_t RQ, uint32_t WAITN>
struct DeviceIO {
    static constexpr uint32_t BYTES = RQ * 16;
    uint32_t ring;        // shared-space byte address of the lane's ring (BYTES bytes, BYTES-aligned)
    uint32_t rot;         // 16 * (lane & 7): rotates the ring index so that lanes in step hit different banks
    const uint4* gbase;   // the frame's 16-byte aligned base
    uint32_t qlim;        // quads readable from gbase (beyond: zeros)
    uint32_t fq;          // next quad to request
    uint32_t wp;          // ring byte offset (unmasked) of the next word of the register window

    __device__ __forceinline__ void issue(uint32_t q) {
        const uint32_t dst = ring | (((q << 4) + rot) & (BYTES - 16u));
        const bool in = q < qlim;
        const uint4* src = gbase + (in ? q : 0u);
        const uint32_t sz = in ? 16u : 0u;  // src-size 0: the destination is zero-filled
        // .cg: straight from L2.  32 lanes ask for 32 different lines; letting them allocate in L1 (.ca) costs the
        // load/store unit far more than the second half of each 32-byte sector being fetched again later.
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
    }
    __device__ __forceinline__ uint32_t word(uint32_t wi) const {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(ring | (((wi << 2) + rot) & (BYTES - 4u))) : "memory");
        return __byte_perm(v, 0, 0x0123);
    }
    __device__ __forceinline__ void seek_next(uint32_t wi) { wp = (wi << 2) + rot; }
    __device__ __forceinline__ uint32_t next_raw() {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(ring | (wp & (BYTES - 4u))) : "memory");
        wp += 4;
        return v;
    }
    // Random access (headers, slow codes): the ring covers quads [bitpos >> 7, (bitpos >> 7) + RQ) on return.
    __device__ __forceinline__ void ensure(uint32_t bitpos) {
        const uint32_t q0 = bitpos >> 7, need = q0 + RQ;
        if (fq < need) {
            if (fq < q0) fq = q0;
            while (fq < need) { issue(fq); fq++; }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    // Before a read of at most 16 bytes from bitpos on (a header field, a single code, a window seat): nothing to
    // do if the steady-state refill is far enough ahead — at most max(WAITN, 4) quads behind its front are still
    // in flight, see prefetch_group() and prefetch_run() — else a blocking refill.
    __device__ __forceinline__ void ensure_near(uint32_t bitpos) {
        if (fq < (bitpos >> 7) + 2u + (WAITN > 4u ? WAITN : 4u)) ensure(bitpos);
    }
    // Steady state, once per group of eight codes.  A group consumes at most 256 bits = 2 quads (C2: 0.36 on
    // average): one predicated copy per group keeps the ring ahead of light streams, a second one — behind a
    // branch that light streams never take — keeps it ahead of dense ones (large Rice parameters: a quad per
    // group and more).  The group needs quads up to (bitpos >> 7) + 3; copies of the last WAITN light groups may
    // still be in flight.  Always true here (the host harness's policy shares the signature).
    __device__ __forceinline__ bool prefetch_group(uint32_t bitpos) {
        const uint32_t q0 = bitpos >> 7;
        if (fq < q0 + RQ) { issue(fq); fq++; }
        if (fq < q0 + RQ) {  // a dense stretch: a second quad this group (more than two only after a jump of the cursor)
            issue(fq); fq++;
            const bool more = fq < q0 + RQ;
            while (fq < q0 + RQ) { issue(fq); fq++; }
            asm volatile("cp.async.commit_group;" ::: "memory");
            // A group of two quads waits for everything older, so that the copies in flight never exceed four
            // quads (this pair plus at most one from each of two later light groups): the RQ - 4 quads from the
            // cursor on, which is what a group reads, have always landed.
            // (A ring with room for two quads from each of WAITN groups beyond the four being read needs none of this.)
            if (more) asm volatile("cp.async.wait_group 0;" ::: "memory");
            else if (2u * WAITN + 4u <= RQ) asm volatile("cp.async.wait_group %0;" ::"n"(WAITN) : "memory");
            else asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group %0;" ::"n"(WAITN) : "memory");
        }
        return true;
    }
    // Steady state of the index lane, once per run of groups that consumes at most `quads` quads from bitpos on: the
    // ring is topped up to RQ quads from the cursor's quad q0 in one commit group.  The run reads quads q0 ..
    // q0 + quads + 1 (the last one for the window's look-ahead word).  What it reads has landed: every older commit
    // group has after wait_group 1, and this one's n quads are the newest, from q0 + RQ - n on, beyond the run's
    // reach while n + quads + 2 <= RQ.  At most max(WAITN, 4) quads are left in flight, as ensure_near() assumes;
    // a run that has to issue more (a dense stretch, a jump of the cursor) waits for all of them.
    // The first two copies are predicated, not branched over: a run of light codes (C2: 1.5 quads) needs no more.
    __device__ __forceinline__ void prefetch_run(uint32_t bitpos, uint32_t quads) {
        const uint32_t q0 = bitpos >> 7, need = q0 + RQ;
        if (fq < q0) fq = q0;
        const uint32_t f0 = fq;
#pragma unroll
        for (int i = 0; i < 2; i++) {
            if (fq < need) { issue(fq); fq++; }
        }
        static_assert(2u <= (WAITN > 4u ? WAITN : 4u), "two copies may stay in flight");
        if (fq < need) {
            while (fq < need) { issue(fq); fq++; }
            asm volatile("cp.async.commit_group;" ::: "memory");
            const uint32_t n = fq - f0;
            if (n <= (WAITN > 4u ? WAITN : 4u) && n + quads + 2u <= RQ) asm volatile("cp.async.wait_group 1;" ::: "memory");
            else asm volatile("cp.async.wait_group 0;" ::: "memory");
        } else {  // n <= 2: the same test, decided at compile time
            asm volatile("cp.async.commit_group;" ::: "memory");
            if (quads + 4u <= RQ) asm volatile("cp.async.wait_group 1;" ::: "memory");
            else asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
    }
    __device__ __forceinline__ void open(uint32_t ring_addr, uint32_t lane, const uint8_t* bytes, uint64_t buf_bytes,
                                         uint64_t byte_offset) {
        ring = ring_addr;
        rot = (lane & 7u) << 4;
        fq = 0;
        wp = 0;
        const uint64_t aligned = byte_offset & ~15ull;
        gbase = reinterpret_cast<const uint4*>(bytes + aligned);
        qlim = (uint32_t)min((buf_bytes - aligned) >> 4, (uint64_t)0x1ffffffu);
    }
    __device__ __forceinline__ void close() { asm volatile("cp.async.wait_all;" ::: "memory"); }
    __device__ __forceinline__ void open_idle(uint32_t ring_addr, uint32_t lane, const uint8_t* bytes) {
        ring = ring_addr;
        rot = (lane & 7u) << 4;
        fq = 0;
        wp = 0;
        gbase = reinterpret_cast<const uint4*>(bytes);
        qlim = 0;
    }
};


// ---------------------------------------------------------------------------------
// Device IO policy of a lane, TMA flavour: a ring of two CHUNK-byte halves in shared memory, each filled by
// one bulk copy (`cp.async.bulk`, SASS UBLKCP) that signals the half's own mbarrier
// ---------------------------------------------------------------------------------
// MEASUREMENT BUILD ONLY (-DCLX_RING_TMA, CLX_RING_TMA=1 in claxon_b200/_build.py): bit-exact (all GPU parity
// tests pass with it) but 18 % slower than the cp.async ring above — a bulk copy takes uniform-register operands,
// so the compiler serves 32 lanes with 32 sources through a loop of ~9 instructions per lane, against one LDGSTS
// for the whole warp (profiles/ab_ring_tma_r02.json vs ab_ring_cpasync_r02.json).  Kept so that the comparison can
// be repeated; the product library is built without it.  (Those figures predate the index lane's runs, for which the
// index ring's chunks went from 128 to 256 bytes; that build compiles but has not been re-run since.)
// Chunk c of the frame (CHUNK bytes from its 16-byte aligned base) lives in half c & 1.  A half is re-armed
// only after the cursor has left the chunk it held, so at most one copy per half is ever outstanding and the
// parity to wait for simply alternates.  Reads past the end of the byte buffer see the buffer's last chunk
// instead (never a fault); running past a frame's own bytes is detected by position, as everywhere.
template <uint32_t CHUNK>
struct TmaIO {
    static constexpr uint32_t BYTES = 2 * CHUNK;
    static constexpr uint32_t CB = CHUNK * 8;     // bits per chunk
    static constexpr uint32_t LANE_BYTES = BYTES + 16;  // ring + two mbarriers; 16 bytes of bank skew between lanes
    uint32_t ring;         // shared-space address of the lane's ring (16-byte aligned); the mbarriers follow it
    const uint8_t* gbase;  // the frame's 16-byte aligned base
    uint32_t clim;         // highest chunk index that lies inside the byte buffer
    uint32_t creq;         // chunks below creq have been requested (the ring holds creq - 2 and creq - 1)
    uint32_t cready;       // chunks below cready have landed
    uint32_t phase;        // bit h: the parity half h's mbarrier completes next
    uint32_t wp;           // byte offset (unmasked) of the next word of the register window
    bool live;

    __device__ __forceinline__ void request(uint32_t c) {
        const uint32_t h = c & 1u;
        const uint32_t bar = ring + BYTES + h * 8u, dst = ring + h * CHUNK;
        const uint8_t* src = gbase + (size_t)min(c, clim) * CHUNK;
        // order this thread's earlier generic-proxy reads of the half before the async-proxy write
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "n"(CHUNK) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                     "l"(src), "n"(CHUNK), "r"(bar)
                     : "memory");
    }
    __device__ __forceinline__ void wait(uint32_t c) {
        const uint32_t h = c & 1u;
        const uint32_t bar = ring + BYTES + h * 8u, parity = (phase >> h) & 1u;
        uint32_t done;
        do {
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(done)
                : "r"(bar), "r"(parity)
                : "memory");
        } while (!done);
        phase ^= 1u << h;
    }
    __device__ __forceinline__ uint32_t word(uint32_t wi) const {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(ring + ((wi << 2) & (BYTES - 4u))) : "memory");
        return __byte_perm(v, 0, 0x0123);
    }
    __device__ __forceinline__ void seek_next(uint32_t wi) { wp = wi << 2; }
    __device__ __forceinline__ uint32_t next_raw() {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(ring + (wp & (BYTES - 4u))) : "memory");
        wp += 4;
        return v;
    }
    // Random access (headers, slow codes): on return the chunk of bitpos has landed, and the next one too if
    // bitpos is within 32 bytes of it (no caller reads further than that without asking again).
    __device__ __forceinline__ void ensure(uint32_t bitpos) {
        if (!live) return;
        const uint32_t c0 = bitpos / CB, c1 = (bitpos + 256u) / CB;
        if (creq < c0) {  // the cursor jumped past everything requested: drain, then start over at its chunk
            while (cready < creq) { wait(cready); cready++; }
            creq = cready = c0;
        }
        while (creq < c0 + 2u) { request(creq); creq++; }
        while (cready <= c1) { wait(cready); cready++; }
    }
    __device__ __forceinline__ void ensure_near(uint32_t bitpos) {
        if (creq < bitpos / CB + 2u || cready <= (bitpos + 256u) / CB) ensure(bitpos);
    }
    // Steady state, once per group of eight codes (at most 256 bits, plus the window's three words of look-ahead).
    __device__ __forceinline__ bool prefetch_group(uint32_t bitpos) {
        const uint32_t c0 = bitpos / CB, c1 = (bitpos + 384u) / CB;
        if (live && creq < c0 + 2u) {
            if (creq < c0 + 1u) ensure(bitpos);  // (after a jump of the cursor)
            else { request(creq); creq++; }      // the cursor has just left chunk c0 - 1: its half takes chunk c0 + 1
        }
        while (live && cready <= c1) { wait(cready); cready++; }
        return true;
    }
    // Once per run of groups that consumes at most `quads` quads from bitpos on (the window's look-ahead word
    // included, it reads up to quad (bitpos >> 7) + quads + 1): needs a CHUNK of at least (quads + 2) * 16 bytes.
    __device__ __forceinline__ void prefetch_run(uint32_t bitpos, uint32_t quads) {
        const uint32_t c0 = bitpos / CB, c1 = (((bitpos >> 7) + quads + 1u) << 7) / CB;
        if (live && creq < c0 + 2u) {
            if (creq < c0 + 1u) ensure(bitpos);
            else { request(creq); creq++; }
        }
        while (live && cready <= c1) { wait(cready); cready++; }
    }
    // No copy into this CTA's shared memory may be in flight when the CTA retires.
    __device__ __forceinline__ void close() {
        while (cready < creq) { wait(cready); cready++; }
    }
    __device__ __forceinline__ void open_idle(uint32_t ring_addr, uint32_t, const uint8_t* bytes) {
        ring = ring_addr;
        gbase = bytes;
        clim = 0; creq = 0; cready = 0; phase = 0; wp = 0;
        live = false;
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(ring + BYTES) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(ring + BYTES + 8u) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // (after open_idle(), which initialised the lane's mbarriers)
    __device__ __forceinline__ void open(uint32_t ring_addr, uint32_t, const uint8_t* bytes, uint64_t buf_bytes, uint64_t byte_offset) {
        ring = ring_addr;
        const uint64_t aligned = byte_offset & ~15ull;
        gbase = bytes + aligned;
        const uint64_t chunks = (buf_bytes - aligned) / CHUNK;  // the buffer is padded: at least one
        clim = (uint32_t)min(chunks - 1, (uint64_t)0x3fffffu);
        creq = 0; cready = 0; wp = 0;
        live = true;
    }
};

// ---------------------------------------------------------------------------------
// Kernel 1: index pass, one lane per frame
// ---------------------------------------------------------------------------------
constexpr uint32_t IDX_RQ = 16;
#ifdef CLX_RING_TMA
using IndexIO = TmaIO<256>;  // a run of IndexLane::RUN groups reads up to 10 quads: 160 bytes must fit one chunk and the next
#else
using IndexIO = DeviceIO<IDX_RQ, 6>;
#endif

__global__ void __launch_bounds__(32)
index_frames_kernel(const uint8_t* __restrict__ bytes, uint64_t buf_bytes, const clx_frame_desc* __restrict__ descs,
                    uint32_t n_frames, clx_frame_result* __restrict__ results, SeqParams* __restrict__ params, uint32_t CH,
                    int* __restrict__ need_generic) {
#ifdef CLX_RING_TMA
    __shared__ __align__(16) uint8_t s_ring[32][IndexIO::LANE_BYTES];
#else
    __shared__ __align__(256) uint4 s_ring[32][IDX_RQ];
#endif
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t fidx = blockIdx.x * 32 + lane;
    const bool live = fidx < n_frames;

    IndexLane<IndexIO> L;
    const uint32_t ring = (uint32_t)__cvta_generic_to_shared(&s_ring[lane][0]);
    L.rc.io.open_idle(ring, lane, bytes);
    if (live) {
        const clx_frame_desc d = descs[fidx];
        L.rc.io.open(ring, lane, bytes, buf_bytes, d.byte_offset);
        L.init(d, params + (size_t)fidx * CH, CH);
    } else {
        clx_frame_desc d = {};
        L.init(d, params, CH);
        L.mode = SEQ_DONE;
        L.rc.ok = true;
    }
    while (__any_sync(0xffffffffu, !L.done())) {
        // the steady state, a tight loop of its own: every lane of the warp steps over a run of up to RUN groups of
        // eight codes (fewer at the end of its partition)
        while (__all_sync(0xffffffffu, L.fast_ready())) L.run();
        // anything else (headers, partition switches, long codes, lanes that are done): one mixed step
        if (L.fast_ready()) L.run();
        else if (!L.done()) L.slow_step();
        __syncwarp();
    }
    L.rc.io.close();
    if (live) {
        clx_frame_result res;
        res.status = L.ok() ? (int32_t)CLX_OK : (int32_t)CLX_INTERNAL_NEED_GENERIC;
        res.consumed = 0;  // set by the lane that decodes the frame's last subframe
        results[fidx] = res;
        if (!L.ok()) *need_generic = 1;
    }
}

// ---------------------------------------------------------------------------------
// Kernel 2: entropy decode + prediction + wasted shift + decorrelation, one lane per subframe
// ---------------------------------------------------------------------------------
#ifndef CLX_DEC_WARPS
#define CLX_DEC_WARPS 2  // warps per decode CTA (1 and 4 were measured too: profiles/SUMMARY_r02.md)
#endif
constexpr int DEC_WARPS = CLX_DEC_WARPS;
constexpr uint32_t DEC_RQ = 8;
#ifdef CLX_RING_TMA
using SubIO = TmaIO<64>;
#else
using SubIO = DeviceIO<DEC_RQ, 3>;
#endif

// One trip of the recurrence for U consecutive samples.  v[0..TAPS) = history (oldest first),
// v[TAPS+i] = sample i of this trip.  Terms that only involve history are summed first, the terms
// with fresh samples last, most recent last — the serial chain per sample is one multiply-add,
// the shift and the residual add.  ACC = long long is the reference's arithmetic verbatim; ACC = int
// is the same recurrence in wrapping 32-bit arithmetic, bit-identical whenever
// sum|coef| * max|sample| < 2^31 — which is re-checked against the samples actually produced.
template <int TAPS, int U, typename ACC>
__device__ __forceinline__ void seq_trip(int32_t (&v)[TAPS + U], const int32_t (&c)[TAPS], const int32_t* r, uint32_t shift) {
    ACC part[U];
#pragma unroll
    for (int i = 0; i < U; i++) {
        ACC acc = 0;
#pragma unroll
        for (int j = 0; j < TAPS; j++)
            if (i + TAPS - 1 - j < TAPS) acc += (ACC)c[j] * (ACC)v[i + TAPS - 1 - j];
        part[i] = acc;
    }
#pragma unroll
    for (int i = 0; i < U; i++) {
        ACC acc = part[i];
#pragma unroll
        for (int j = TAPS - 1; j >= 0; j--)
            if (i + TAPS - 1 - j >= TAPS) acc += (ACC)c[j] * (ACC)v[i + TAPS - 1 - j];
        v[TAPS + i] = (int32_t)(acc >> shift) + r[i];
    }
}

// Where the samples of a tile row (= a lane = a subframe) go; shared memory, one per lane.  Rows 2p and 2p+1
// are neighbouring channels of one frame when the batch has at least two channel slots — `ca` on the even
// row is then the frame's stereo mode if the pair is its (channel 0, channel 1) — and two unrelated mono
// frames otherwise.
struct __align__(16) SeqRow {
    int32_t* out;   // subframe's first output element (nullptr: idle row)
    uint32_t bs;    // block size
    uint32_t meta;  // bit 0: 16-byte stores allowed; bits 8-15: wasted bits; bits 16-19 (even rows): 8 left/side,
                    // 9 side/right, 10 mid/side, 0 independent
};

__device__ __forceinline__ uint32_t seq_tile_word(uint32_t row, uint32_t col) {
    return row * 32 + ((((col >> 2) ^ (row & 7)) << 2) | (col & 3));
}
__device__ __forceinline__ void seq_store_vec(int32_t* out, uint32_t bs, bool vec, uint32_t g, const int4& v) {
    if (out == nullptr || g >= bs) return;
    if (vec && g + 4 <= bs) *reinterpret_cast<int4*>(out + g) = v;
    else {
        out[g] = v.x;
        if (g + 1 < bs) out[g + 1] = v.y;
        if (g + 2 < bs) out[g + 2] = v.z;
        if (g + 3 < bs) out[g + 3] = v.w;
    }
}
__device__ __forceinline__ int4 shl4(const int4& v, uint32_t s) {
    return make_int4((int32_t)((uint32_t)v.x << s), (int32_t)((uint32_t)v.y << s), (int32_t)((uint32_t)v.z << s),
                     (int32_t)((uint32_t)v.w << s));
}
// mid/side -> left/right (src/frame.rs:371-389).  The reference computes m2 = (mid*2)|(side&1) and
// (m2 +- side)/2 in wrapping i32; with no wrap (|mid|, |side| < 2^29, checked by the caller against
// the samples produced) that is mid + (side>>1) + (side&1) and mid - (side>>1), floor shifts.
__device__ __forceinline__ void mid_side(int32_t& a, int32_t& b) {
    const int32_t h = b >> 1;
    const int32_t l = a + b - h;  // side - (side >> 1) = (side >> 1) + (side & 1)
    b = a - h;
    a = l;
}

// Writes a quarter of the warp's 32x32 tile (steps [g0, g0+32) of rows 8q .. 8q+7) to global memory: wasted
// bits (src/subframe.rs:216-225), decorrelation (src/frame.rs:319-389), planar i32.  Eight lanes take the eight
// 16-byte vectors of a row pair (rows 2p, 2p+1), so each store instruction of the warp covers four whole
// 128-byte lines — scattering the lanes over more rows costs the load/store unit a wavefront per line.
// CHECKED = false is for tiles wholly inside every active row with 16-byte stores allowed everywhere.
template <bool CHECKED>
__device__ __forceinline__ void seq_flush_quarter(const int32_t* tile, const SeqRow* rows, uint32_t g0, uint32_t q, uint32_t lane,
                                                  bool any_wasted) {
    const uint32_t grp = lane & 7;
    const uint32_t r0 = (4 * q + (lane >> 3)) * 2, r1 = r0 + 1;
    const uint32_t g = g0 + grp * 4;
    const SeqRow i0 = rows[r0], i1 = rows[r1];
    int4 a = *reinterpret_cast<const int4*>(tile + r0 * 32 + ((grp ^ (r0 & 7)) << 2));
    int4 b = *reinterpret_cast<const int4*>(tile + r1 * 32 + ((grp ^ (r1 & 7)) << 2));
    if (any_wasted) { a = shl4(a, (i0.meta >> 8) & 0xffu); b = shl4(b, (i1.meta >> 8) & 0xffu); }
    const uint32_t ca = (i0.meta >> 16) & 15u;
    if (ca == 10) {
        mid_side(a.x, b.x); mid_side(a.y, b.y); mid_side(a.z, b.z); mid_side(a.w, b.w);
    } else if (ca == 8) {  // left/side (src/frame.rs:319-334)
        b.x = (int32_t)((uint32_t)a.x - (uint32_t)b.x); b.y = (int32_t)((uint32_t)a.y - (uint32_t)b.y);
        b.z = (int32_t)((uint32_t)a.z - (uint32_t)b.z); b.w = (int32_t)((uint32_t)a.w - (uint32_t)b.w);
    } else if (ca == 9) {  // side/right (src/frame.rs:345-360)
        a.x = (int32_t)((uint32_t)a.x + (uint32_t)b.x); a.y = (int32_t)((uint32_t)a.y + (uint32_t)b.y);
        a.z = (int32_t)((uint32_t)a.z + (uint32_t)b.z); a.w = (int32_t)((uint32_t)a.w + (uint32_t)b.w);
    }
    if (CHECKED) {
        seq_store_vec(i0.out, i0.bs, (i0.meta & 1u) != 0, g, a);
        seq_store_vec(i1.out, i1.bs, (i1.meta & 1u) != 0, g, b);
    } else {
        if (i0.out != nullptr) *reinterpret_cast<int4*>(i0.out + g) = a;
        if (i1.out != nullptr) *reinterpret_cast<int4*>(i1.out + g) = b;
    }
}
template <bool CHECKED>
__device__ __forceinline__ void seq_flush(const int32_t* tile, const SeqRow* rows, uint32_t g0, uint32_t lane, bool any_wasted) {
    __syncwarp();
#pragma unroll
    for (uint32_t i = 0; i < 4; i++) seq_flush_quarter<CHECKED>(tile, rows, g0, i, lane, any_wasted);
    __syncwarp();
}

// ---- shared-memory accesses by 32-bit shared-space address (no generic-pointer arithmetic in the hot loop) ----
__device__ __forceinline__ int4 lds128(uint32_t addr) {
    int4 v;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, int32_t a, int32_t b, int32_t c, int32_t d) {
    asm volatile("st.shared.v4.s32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// The common case of seq_flush_quarter, straight-line: every lane of the warp active, every row 16-byte
// aligned, no wasted bits, one stereo mode UCA (0 = none, 10 = mid/side) for every row pair, tile wholly
// inside every row.
//   tile_s: shared address of the tile to write out;  outp_s: shared address of the warp's 32 row pointers;
//   lc0 / lc1: the lane's constant offsets into the tile for rows (2p, 2p+1) of its quarter (see decode_rows).
template <int UCA>
__device__ __forceinline__ void flush_quarter_fast(uint32_t tile_s, uint32_t outp_s, uint32_t g0, uint32_t quarter, uint32_t lane,
                                                   uint32_t lc0, uint32_t lc1) {
    const uint32_t a0 = tile_s + quarter * 1024u + lc0;
    const int4 a = lds128(a0);
    const int4 b = lds128(a0 + lc1);
    unsigned long long p0, p1;  // rows 2 * (4 * quarter + (lane >> 3)) and the next
    asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(p0), "=l"(p1) : "r"(outp_s + quarter * 64u + (lane >> 3) * 16u) : "memory");
    int4 oa = a, ob = b;
    if (UCA == 10) {  // src/frame.rs:371-389, see mid_side()
        const int32_t hx = b.x >> 1, hy = b.y >> 1, hz = b.z >> 1, hw = b.w >> 1;
        oa = make_int4(a.x + b.x - hx, a.y + b.y - hy, a.z + b.z - hz, a.w + b.w - hw);
        ob = make_int4(a.x - hx, a.y - hy, a.z - hz, a.w - hw);
    }
    const uint32_t off = (g0 + (lane & 7u) * 4u) * 4u;  // bytes
    *reinterpret_cast<int4*>(p0 + off) = oa;
    *reinterpret_cast<int4*>(p1 + off) = ob;
}

// The body of a subframe lane: residuals from the lane's own Rice decoder, recurrence, tile, flush.
// Every lane of the warp advances over the same sample index t (lanes whose block is shorter idle at the
// end), so the 32x32 tile fills row by row in step and is flushed as whole lines.
//   tile_s: shared address of the warp's two tiles (8 KB, 8 KB-aligned: the other tile is `addr ^ 4096`).
//   FMODE: 0 = general flush; 1 / 2 = flush_quarter_fast applies, without stereo decorrelation / mid-side.
template <int TAPS, int U, typename ACC, int FMODE>
__device__ __forceinline__ void decode_rows(SubLane<SubIO>& L, uint32_t bs, uint32_t order, uint32_t shift,
                                            const SeqParams* __restrict__ sp, bool active, int32_t* tile, uint32_t tile_s,
                                            const SeqRow* pr, uint32_t outp_s, uint32_t lane, bool all_vec,
                                            bool any_wasted, int32_t& smin, int32_t& smax) {
    int32_t c[TAPS], h[TAPS];  // c[j] multiplies s[t-1-j]; h[j] = s[t-1-j]
#pragma unroll
    for (int j = 0; j < TAPS; j++) {
        c[j] = (active && (uint32_t)j < order) ? (int32_t)sp->coefs[j] : 0;
        // Opaque to the optimiser: otherwise the i16 -> i64 promotion is folded into a full 64-bit
        // multiply (3 instructions) instead of one signed 32x32+64 IMAD.WIDE per tap.
        asm volatile("" : "+r"(c[j]));
        h[j] = 0;
    }
    const uint32_t max_bs = __reduce_max_sync(0xffffffffu, active ? bs : 0u);
    const uint32_t min_bs = __reduce_min_sync(0xffffffffu, active ? bs : 0xffffffffu);
    const uint32_t max_order = __reduce_max_sync(0xffffffffu, active ? order : 0u);
    const uint32_t head_end = min(max_bs, (max_order + 7u) & ~7u);  // whole groups of eight
    const uint32_t bulk_end = min_bs > head_end ? head_end + ((min_bs - head_end) & ~7u) : head_end;

    // Samples are staged in one of two 32x32 tiles; while a tile fills (four trips of 8 samples), the
    // previous one is written out a quarter per trip, so that its shared-memory loads, the
    // decorrelation and its global stores interleave with the decode of the next samples.
    uint32_t fill_s = tile_s;  // the tile being filled; the other one is fill_s ^ 4096
    bool have_drain = false;
    auto tile_ptr = [&](uint32_t s_addr) { return tile + ((s_addr - tile_s) >> 2); };

    auto guarded = [&](uint32_t t0, uint32_t t1) {  // one sample at a time, every condition checked
        for (uint32_t t = t0; t < t1; t++) {
            const bool inside = active && t < bs;
            int32_t val = 0;
            if (inside) {
                if (t < order) val = sp->warm[t];
                else {
                    const int32_t r = L.next();
                    long long acc = 0;
#pragma unroll
                    for (int j = 0; j < TAPS; j++) acc += (long long)c[j] * (long long)h[j];
                    val = r + (sizeof(ACC) == 8 ? (int32_t)(acc >> shift) : (int32_t)((int32_t)acc >> shift));
                }
                smin = min(smin, val);
                smax = max(smax, val);
            }
#pragma unroll
            for (int j = TAPS - 1; j > 0; j--) h[j] = h[j - 1];
            h[0] = val;
            int32_t* fill = tile_ptr(fill_s);
            fill[seq_tile_word(lane, t & 31)] = val;
            if ((t & 31) == 31) seq_flush<true>(fill, pr, t - 31, lane, any_wasted);
        }
    };
    guarded(0, head_end);
    if (bulk_end > head_end) {
        int32_t v[TAPS + U];
#pragma unroll
        for (int j = 0; j < TAPS; j++) v[j] = h[TAPS - 1 - j];
        const uint32_t l7 = lane & 7u, l3 = lane >> 3;
        const uint32_t row_off = lane * 128u;  // the lane's row inside a tile
        // flush_quarter_fast: rows r0 = 2 * (4 * quarter + l3) and r0 + 1; r0 & 7 = 2 * l3 whatever the quarter
        const uint32_t lc0 = l3 * 256u + ((l7 ^ (2u * l3)) << 4);
        const uint32_t lc1 = 128u + (((l7 ^ (2u * l3 + 1u)) << 4) - ((l7 ^ (2u * l3)) << 4));

        // The loop is software-pipelined: a trip predicts the eight samples whose residuals the PREVIOUS trip
        // decoded, and decodes — speculatively and branch-free, see RiceCursor::spec_group — the residuals of the
        // next eight, in the same basic block: two independent dependency chains, one bound by the ALU pipe (bit
        // scan), the other by the multiply-add pipe (recurrence), for the instruction scheduler to interleave.
        int32_t rA[8], rB[8];
        // residuals of the next eight samples by the ordinary route (the start, and whenever speculation fails)
        auto produce = [&](int32_t (&dst)[8], bool try_fast) {
            bool got = false;
            if (try_fast) {
                if (!L.fast()) L.prepare();  // partition switch, window seat
                if (L.fast()) got = L.fast_group(dst);
            }
            if (!got) {  // a partition boundary inside the group, a code longer than the window, verbatim ...
                int32_t slow_e[8];  // indexed by a loop variable on purpose: local memory, touched on this slow path only
#pragma unroll 1
                for (int i = 0; i < 8; i++) slow_e[i] = L.next();
#pragma unroll
                for (int i = 0; i < 8; i++) dst[i] = slow_e[i];
            }
        };
        // prediction of samples t .. t+7 from their residuals, exactness bounds, staging in the tile
        auto consume = [&](const int32_t (&r)[8], uint32_t t) {
            // the lane's two 16-byte slots of this trip: columns (t & 31) .. +3 and +4 .. +7, swizzled by the row
            const uint32_t slot0 = fill_s + row_off + (((((t >> 2) & 6u)) ^ l7) << 4);
#pragma unroll
            for (int half = 0; half < 8 / U; half++) {
                seq_trip<TAPS, U, ACC>(v, c, r + half * U, shift);
#pragma unroll
                for (int i = 0; i < U; i += 2) {
                    smax = __vimax3_s32(smax, v[TAPS + i], v[TAPS + i + 1]);
                    smin = __vimin3_s32(smin, v[TAPS + i], v[TAPS + i + 1]);
                }
#pragma unroll
                for (int q = 0; q < U / 4; q++)
                    sts128(slot0 ^ ((uint32_t)(half * (U / 4) + q) << 4), v[TAPS + 4 * q], v[TAPS + 4 * q + 1], v[TAPS + 4 * q + 2],
                           v[TAPS + 4 * q + 3]);
#pragma unroll
                for (int j = 0; j < TAPS; j++) v[j] = v[j + U];
            }
        };
        // a quarter of the previous tile goes out; a full tile becomes the one to write out
        auto after = [&](uint32_t t) {
            if (have_drain) {  // a tile inside [head_end, bulk_end) lies inside every active row
                const uint32_t g0 = (t & ~31u) - 32, quarter = (t >> 3) & 3;
                if (FMODE != 0) flush_quarter_fast<FMODE == 2 ? 10 : 0>(fill_s ^ 4096u, outp_s, g0, quarter, lane, lc0, lc1);
                else if (all_vec) seq_flush_quarter<false>(tile_ptr(fill_s ^ 4096u), pr, g0, quarter, lane, any_wasted);
                else seq_flush_quarter<true>(tile_ptr(fill_s ^ 4096u), pr, g0, quarter, lane, any_wasted);
            }
            if (((t + 8) & 31) == 0) {
                __syncwarp();
                fill_s ^= 4096u;
                have_drain = true;
            }
        };
        // MP: some subframe of the warp has a partition boundary ahead (its own instance of the loop, so that warps
        // of single-partition subframes do not even look)
        // COMPACT: the bodies that warps of mixed batches end up in (general flush: irregular rows, or the i64
        // accumulator).  An SM then runs several DIFFERENT bodies at once and its 32 KB instruction cache holds
        // the loops of all of them only if each is small: one trip per iteration (the residuals are copied
        // instead of alternating between two register sets), one code per window refill, one instance for
        // single- and multi-partition warps.  The regular bodies (FMODE != 0: whole batches of one shape, one
        // loop on every SM) keep the unrolled, specialised form.
        constexpr bool COMPACT = FMODE == 0;
        uint32_t nc_fixed = 1;
        auto step = [&](auto mp, const int32_t (&cons)[8], int32_t (&prod)[8], uint32_t t) {
            if (decltype(mp)::value && active && !L.fast()) L.quick_prepare();  // a partition header, from the window
            bool good;
            if (COMPACT) { good = L.template spec_group<1>(prod); consume(cons, t); }
            else {
                // codes per window refill: what every lane on the fast path allows (by its partition's Rice parameter);
                // fixed for the whole loop when no lane has a partition boundary ahead
                const uint32_t nc = decltype(mp)::value ? __reduce_min_sync(0xffffffffu, L.spec_cap()) : nc_fixed;
                if (nc == 2) { good = L.template spec_group<2>(prod); consume(cons, t); }
                else { good = L.template spec_group<1>(prod); consume(cons, t); }
            }
            if (!good && active) produce(prod, true);  // rare
            after(t);
        };
        if (active) produce(rA, true);
        uint32_t t = head_end;
        auto run = [&](auto mp) {
            if (COMPACT) {
                while (t + 8 < bulk_end) {
                    step(mp, rA, rB, t);
#pragma unroll
                    for (int i = 0; i < 8; i++) rA[i] = rB[i];
                    t += 8;
                }
                consume(rA, t);
                return;
            }
            while (t + 16 < bulk_end) {
                step(mp, rA, rB, t);
                step(mp, rB, rA, t + 8);
                t += 16;
            }
            if (t + 8 < bulk_end) {
                step(mp, rA, rB, t);
                t += 8;
                consume(rB, t);
            } else consume(rA, t);
        };
        if (COMPACT || __any_sync(0xffffffffu, active && L.rc.parts_left != 0)) run(std::true_type{});
        else {
            nc_fixed = __reduce_min_sync(0xffffffffu, active ? L.last_cap() : 2u);
            run(std::false_type{});
        }
        after(t);
        if (have_drain) {  // whatever of the last full tile has not been written yet (re-writing a quarter is harmless)
            const uint32_t g0 = (bulk_end & ~31u) - 32;
#pragma unroll
            for (uint32_t i = 0; i < 4; i++) seq_flush_quarter<true>(tile_ptr(fill_s ^ 4096u), pr, g0, i, lane, any_wasted);
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < TAPS; j++) h[j] = v[TAPS - 1 - j];
    }
    guarded(bulk_end, max_bs);
    if (max_bs & 31) seq_flush<true>(tile_ptr(fill_s), pr, max_bs & ~31u, lane, any_wasted);
}

// Two instances, launched back to back: GROUP 0 takes the warps whose largest predictor order is at most 12 (with
// an 8-tap and a 12-tap body: every warp of a batch of mixed orders runs at once), GROUP 1 the warps with orders
// up to 32 (non-subset streams), whose body needs half as many registers again.  A warp does its work in the
// instance of its group and leaves the other at once.
//
// WIDE = true is the second chance of frames whose samples left the range the i32 accumulator is exact for (see
// below): the same rows once more with the reference's i64 arithmetic only.  It looks at nothing unless the first
// pass raised `need_wide`.
template <int GROUP, bool WIDE>
__global__ void __launch_bounds__(DEC_WARPS * 32)
decode_subframes_kernel(const uint8_t* __restrict__ bytes, uint64_t buf_bytes, const clx_frame_desc* __restrict__ descs,
                        uint32_t n_frames, int32_t* __restrict__ out, clx_frame_result* __restrict__ results,
                        const SeqParams* __restrict__ params, uint32_t CH, uint32_t ch_log2, uint32_t n_pwarps,
                        int* __restrict__ need_generic, int* __restrict__ need_wide) {
    __shared__ __align__(8192) int32_t s_tile[DEC_WARPS][2 * 32 * 32];  // two tiles: one fills while the other drains
    __shared__ SeqRow s_rows[DEC_WARPS][32];
    __shared__ __align__(16) int32_t* s_outp[DEC_WARPS][32];
#ifdef CLX_RING_TMA
    __shared__ __align__(16) uint8_t s_ring[DEC_WARPS][32][SubIO::LANE_BYTES];
#else
    __shared__ __align__(128) uint4 s_ring[DEC_WARPS][32][DEC_RQ];
#endif
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t pw = blockIdx.x * DEC_WARPS + warp;  // CH subframe warps per group of 32 frames
    if (pw >= n_pwarps) return;
    if (WIDE && *need_wide == 0) return;
    const uint32_t w = pw >> ch_log2, part = pw & (CH - 1);
    const uint32_t j = part * (32u >> ch_log2) + (lane >> ch_log2);  // frame within the group
    const uint32_t c = lane & (CH - 1);
    const uint32_t f = w * 32 + j;
    int32_t* tile = s_tile[warp];

    bool active = false, narrow_ok = true, last = false;
    uint32_t bs = 0, order = 0, shift = 0, wasted = 0, ca = 0, absum = 0, bit0 = 0, byte_len = 0;
    const SeqParams* sp = params;
    int32_t* sub = nullptr;
    SubLane<SubIO> L;
    const uint32_t ring = (uint32_t)__cvta_generic_to_shared(&s_ring[warp][lane][0]);
    L.rc.io.open_idle(ring, lane, bytes);
    L.init_idle();
    if (f < n_frames && results[f].status == (WIDE ? (int32_t)CLX_INTERNAL_NEED_WIDE : (int32_t)CLX_OK)) {
        const clx_frame_desc d = descs[f];
        if (c < d.n_channels) {
            sp = params + (size_t)f * CH + c;
            active = true;
            last = c + 1 == d.n_channels;
            bs = d.block_size;
            order = (uint32_t)sp->order;
            shift = (uint32_t)sp->shift;
            wasted = (uint32_t)sp->wasted;
            absum = sp->absum;
            ca = d.channel_assignment >= 8 ? d.channel_assignment : 0u;
            sub = out + d.out_offset + (size_t)c * bs;
            uint32_t bits = d.bits_per_sample;  // nominal sample width (one extra bit for a side channel)
            if (d.channel_assignment == 9) bits += (c == 0);
            else if (d.channel_assignment == 8 || d.channel_assignment == 10) bits += (c == 1);
            // valid streams keep |sample| <= 2^(bits-1); anything beyond is caught by the check below
            narrow_ok = ((unsigned long long)absum << (bits - 1)) < (1ull << 31);
            bit0 = (uint32_t)(d.byte_offset & 15) * 8;
            byte_len = d.byte_len;
        }
    }
    if (!__any_sync(0xffffffffu, active)) return;
    const uint32_t max_order = __reduce_max_sync(0xffffffffu, active ? order : 0u);
    const int cls = max_order <= 8 ? 0 : max_order <= 12 ? 1 : 2;
    if ((cls == 2) != (GROUP == 1)) return;
    const bool vec_own = (reinterpret_cast<uintptr_t>(sub) & 15) == 0;
    const bool all_vec = __all_sync(0xffffffffu, !active || vec_own);
    SeqRow* pr = s_rows[warp];
    {
        SeqRow row;
        row.out = sub;
        row.bs = bs;
        row.meta = (vec_own ? 1u : 0u) | (wasted << 8) | ((c == 0 ? ca : 0u) << 16);
        pr[lane] = row;
        s_outp[warp][lane] = sub;
    }
    __syncwarp();

    const bool all_narrow = __all_sync(0xffffffffu, !active || narrow_ok);
    const bool any_wasted = __any_sync(0xffffffffu, active && wasted != 0);
    // flush_quarter_fast: full warp, aligned rows, no wasted bits, and one stereo mode on every row pair
    // (with one channel slot per frame, rows 2p and 2p+1 are unrelated frames: mode 0)
    const uint32_t pair_ca = CH >= 2 ? __shfl_sync(0xffffffffu, ca, lane & ~1u) : 0u;
    const uint32_t ca0 = __shfl_sync(0xffffffffu, pair_ca, 0);
    const bool fast_flush = __all_sync(0xffffffffu, active && vec_own && wasted == 0 && pair_ca == ca0);
    const int fmode = !fast_flush ? 0 : ca0 == 0 ? 1 : ca0 == 10 ? 2 : 0;
    int32_t smin = 0, smax = 0;
    const uint32_t tile_s = (uint32_t)__cvta_generic_to_shared(tile);
    const uint32_t outp_s = (uint32_t)__cvta_generic_to_shared(&s_outp[warp][0]);
#define CLX_ROWS(T, UU, A, F) decode_rows<T, UU, A, F>(L, bs, order, shift, sp, active, tile, tile_s, pr, outp_s, lane, all_vec, any_wasted, smin, smax)
    // straight-line flush variants only where they pay: the i32-accumulator bodies (16-bit audio).  The i64 bodies are
    // what mixed batches run, several per SM at a time; there one body (12 taps, also for warps that would do with
    // 8) beats two that evict each other from the instruction cache.
#define CLX_INT(T, UU)                                 \
    do {                                               \
        if (fmode == 2) CLX_ROWS(T, UU, int, 2);       \
        else if (fmode == 1) CLX_ROWS(T, UU, int, 1);  \
        else CLX_ROWS(T, UU, int, 0);                  \
    } while (0)
    // The i32 accumulator is exact only while sum|coef| * max|sample| < 2^31, which is checked against the samples
    // actually produced.  Streams that keep to their nominal sample width never fail it; a frame whose samples do
    // leave that range is decoded once more by the WIDE instance (the reference's i64 arithmetic).
    const bool narrow = !WIDE && all_narrow;
    if (WIDE) {
        if (active && c == 0) results[f].status = CLX_OK;  // this pass's verdict replaces the first one's
        __syncwarp();
    }
    if (active) {
        L.rc.io.open(ring, lane, bytes, buf_bytes, descs[f].byte_offset);
        L.init(*sp, bs, bit0 + byte_len * 8);
    }
    if (GROUP == 1) {
        if (narrow) CLX_INT(32, 4);
        else CLX_ROWS(32, 4, long long, 0);
    } else if (!narrow) CLX_ROWS(12, 4, long long, 0);  // ONE call site, hence one copy of the body, for both order classes
    else if (cls == 0) CLX_INT(8, 8);
    else CLX_INT(12, 4);
#undef CLX_INT
#undef CLX_ROWS
    if (!active) return;
    // The subframe must end inside the frame; the lane of the last subframe locates the CRC-16 footer
    // (pad bits up to the byte boundary are skipped unchecked, src/frame.rs:744-754).
    const uint32_t end_bit = L.finish();
    L.rc.io.close();
    bool redo = !L.ok();
    if (last && !redo) {
        const uint32_t consumed = ((end_bit - bit0 + 7) >> 3) + 2;
        if (consumed > byte_len) redo = true;
        else results[f].consumed = consumed;
    }
    // The mid/side shortcut (no wrapping intermediate) is exact only while max|sample| << wasted < 2^29 on both
    // channels, again checked on the samples produced; a frame that fails is re-decoded by the generic kernel.
    const uint32_t m = max((uint32_t)smax, 0u - (uint32_t)smin);
    if (narrow && order > 0 && (unsigned long long)absum * m >= (1ull << 31)) {
        if (!redo) results[f].status = CLX_INTERNAL_NEED_WIDE;  // (a frame that needs the generic kernel anyway keeps that mark)
        *need_wide = 1;
    }
    if (ca == 10 && (((unsigned long long)m) << wasted) >= (1ull << 29)) redo = true;
    if (redo) {
        results[f].status = CLX_INTERNAL_NEED_GENERIC;  // takes precedence over NEED_WIDE whatever the order of the writes:
        *need_generic = 1;                              // the WIDE pass only picks up frames still marked NEED_WIDE
    }
}

// ---------------------------------------------------------------------------------
// launch helpers
// ---------------------------------------------------------------------------------
#ifdef CLX_EXPERIMENT
int g_exp_which = 3;
int g_exp_dyn_smem = 0;  // extra dynamic shared memory per decode CTA: lowers occupancy (measurement only)
#endif

size_t seq_scratch_bytes(const CoopPlan& plan, uint32_t n_frames) {
    const uint32_t n_warps = (n_frames + 31) / 32;
    const size_t b = (size_t)n_warps * 32 * plan.channels * sizeof(SeqParams);
    return ((b + 511) & ~(size_t)511) + 512;
}

cudaError_t launch_seq(const uint8_t* d_bytes, uint64_t buf_bytes, const clx_frame_desc* d_descs, uint32_t n_frames,
                       int32_t* d_out, clx_frame_result* d_results, int* d_need_generic, void* d_params,
                       const CoopPlan& plan, cudaStream_t stream, int which) {
#ifdef CLX_EXPERIMENT
    which &= g_exp_which;
#endif
    const uint32_t CH = plan.channels;
    uint32_t ch_log2 = 0;
    while ((1u << ch_log2) < CH) ch_log2++;
    const uint32_t n_warps = (n_frames + 31) / 32;
    SeqParams* params = reinterpret_cast<SeqParams*>(d_params);
    if (which & 1)
        index_frames_kernel<<<n_warps, 32, 0, stream>>>(d_bytes, buf_bytes, d_descs, n_frames, d_results, params, CH,
                                                        d_need_generic);
    if (which & 2) {
        const uint32_t n_pwarps = n_warps * CH;
        dim3 g2((n_pwarps + DEC_WARPS - 1) / DEC_WARPS), b2(DEC_WARPS * 32);
#ifdef CLX_EXPERIMENT
        const size_t dyn = (size_t)g_exp_dyn_smem;
#else
        const size_t dyn = 0;
#endif
#define CLX_DEC(C, W) decode_subframes_kernel<C, W><<<g2, b2, dyn, stream>>>(d_bytes, buf_bytes, d_descs, n_frames, d_out, d_results, params, CH, ch_log2, n_pwarps, d_need_generic, d_need_generic + 2)
        CLX_DEC(0, false); CLX_DEC(1, false); CLX_DEC(0, true); CLX_DEC(1, true);
#undef CLX_DEC
    }
    return cudaGetLastError();
}

}  // namespace clx
