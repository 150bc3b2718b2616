// afsk_rx.cu — receiver path of libafsk_b200.so (sm_100a).
//
// Replaces the compute of Receiver.load (afskmodem.py:420-430) for a batch of independent
// captures with three kernels:
//
//   k_clock   __recoverClockIndex (:322-339): first 4096 frames -> prefix sum in shared memory,
//             every candidate offset scored from 7 prefix taps (closed form of getDiff against
//             the +/-full-scale training cycle) kept in registers along chains of candidates a
//             quarter bit apart, block arg-min with first-index ties.
//   k_demod   __decodeBit (:342-351) + __amplify (:287-296) + getAmplitude (:94-98) for EVERY
//             bit window of every capture: the streaming, HBM-bound kernel.  Persistent CTAs,
//             1-D TMA bulk copies (cp.async.bulk -> UBLKCP) into a multi-stage shared-memory ring
//             fed by a producer warp, mbarrier full/empty hand-off, consumers read 128-bit
//             vectors and reduce each window to a mark/space decision bit and a "quiet" bit with
//             packed 16x2 integer ops and IDP.2A dot products.  Output: 2 bits per window.
//   k_frame   __scanTraining (:386-390) terminator search, the data loop's end detector (:372-378),
//             ECC.decode (:154-163) and __bitsToBytes (:393-399) on the packed bit planes
//             (k_frame_warp: one warp per capture; k_frame: one CTA per capture for very long ones).
//
// All arithmetic is integer and bit-exact with the reference (see DESIGN.md for the algebra).
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <new>
#include <utility>
#include <vector>

#include "afsk_common.cuh"

#ifdef AFSK_DBG_TRACE
// debugging build only: time stamps (ns, %globaltimer) of auxiliary-warp jobs, read back by afsk_dbg_trace_read
__device__ unsigned long long g_trace[1 << 16];
__device__ unsigned int g_trace_n;
__device__ __forceinline__ unsigned long long trace_now()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define AFSK_TRACE_DECL unsigned long long tr__[8]; int trn__ = 0;
#define AFSK_TRACE_MARK if (trn__ < 8) tr__[trn__++] = trace_now();
#define AFSK_TRACE_EMIT(kind)                                                              \
    if ((threadIdx.x & 31) == 0 && ((kind) != 1ull || (blockIdx.x & 15) == 0)) {           \
        const unsigned int slot__ = atomicAdd(&g_trace_n, 1u);                             \
        if (slot__ < (1u << 12)) {                                                         \
            g_trace[slot__ * 10] = (kind);                                                 \
            g_trace[slot__ * 10 + 1] = (unsigned long long)trn__;                          \
            for (int q__ = 0; q__ < 8; q__++) g_trace[slot__ * 10 + 2 + q__] = q__ < trn__ ? tr__[q__] : 0ull; \
        }                                                                                  \
    }
#else
#define AFSK_TRACE_DECL
#define AFSK_TRACE_MARK
#define AFSK_TRACE_EMIT(kind)
#endif

namespace {

constexpr int kConsumerThreads = 256;
constexpr int kDemodThreads = kConsumerThreads + 32;   // + one producer warp
constexpr int kMaxStages = 8;
constexpr int kClockThreads = 128;
constexpr int kClockChain = 35;     // candidates per chain in k_clock
constexpr int kFrameThreads = 128;    // k_gate_scan block; k_frame is templated on its own block size

struct __align__(16) CapDesc {
    int64_t off;         // first sample of the capture (global sample index)
    int64_t n;           // samples in the capture
    int64_t plane_base;  // word offset of the capture's rows in the bit / quiet planes
    int64_t out_off;     // byte offset of the capture's decoded payload
    int32_t bf;          // Receiver.__bit_frames (:277)
    int32_t thr;         // amp_end_threshold clamped to [0, 65537]
    int32_t status0;     // 0 -> decode on the GPU; otherwise the final AFSK_ST_* status
    int32_t group;       // index of the baud group (kernel launch) the capture belongs to
};

struct __align__(16) TileMeta {
    int32_t e0;          // first window's sample offset inside the copy (< 64; the copy starts 16-byte aligned)
    int32_t nwin;        // valid windows in this tile (0 -> nothing to do)
    int32_t thr_bf;      // amp_end * bf : quiet <=> sum|x| < thr_bf
    int32_t gpos;        // position of the tile's capture in the group's capture list
    int64_t word_base;   // plane word receiving window 0 of the tile
    uint32_t want;       // tiles of the tile's capture (fused framing: the capture is complete when all have been reported)
    int32_t pad2;
};

struct DemodParams {
    const int16_t *samples;
    const CapDesc *caps;
    const int32_t *clock;
    const int32_t *gcaps;        // capture ids of this group, ascending
    const int32_t *gtile_first;  // [ng + 1] prefix of tile counts over gcaps
    const int32_t *tile_gpos;    // [total_items] tile -> position of its capture in gcaps
    uint2 *planes;               // {bit word, quiet word} per 32 windows
    int ng;
    int total_items;
    int bf;
    int tpw_log2;     // threads per window = 1 << tpw_log2
    int seg;          // samples per thread segment = ceil(bf / tpw)
    int nv;           // 16-byte vectors each thread reads
    int nt;           // weight-table entries per (part, alignment): nv, or nv - 1 in merge mode
    int merge;        // seg % 8 == 0: head and tail partial vectors are merged into one
    int wt;           // windows per tile = nsub * (kConsumerThreads >> tpw_log2)
    int nsub;         // sub-tiles per tile (general kernel; 1 elsewhere)
    int rot;          // 32-sample segments: rotated vector order (AFSK_NO_ROT=1 turns it off for A/B runs)
    int stage_bytes;
    int stages;
    int l2_hint;      // 1: bulk copies carry an L2 evict-first policy
    int pad_warps;    // padded layout: warps that share the cp.async copies of a tile (1..5)
    // ---- fused mode: auxiliary warps of every CTA recover the clocks and frame the captures of this group
    //      inside the same launch (k_clock / k_frame_warp become jobs hidden under the HBM stream)
    int fused;        // 0: clocks come from k_clock (p.clock); 1: from the auxiliary warps (p.cready)
    int fused_frame;  // 1: the auxiliary warps also run the framing of every capture whose last tile has retired
    uint32_t epoch;   // decode counter of the plan: a clock word is valid iff its tag equals it
    int aux_off;      // byte offset of the AuxSmem block in dynamic shared memory
    uint32_t clk_magic;                  // floor(D / 2bf) == (D * clk_magic) >> clk_shift for D < 2^28
    int clk_shift;
    unsigned long long *cready;          // [B] {clock index, epoch tag}: one 64-bit word per capture
    int32_t *clock_out;                  // [B] clock index as k_clock leaves it (for k_frame / diagnostics)
    uint32_t *tiles_done;                // [ng] consumer-warp arrivals per capture (reset by the framing job)
    uint32_t *ctrl;                      // [2][4] job counters {next clock job}, slot = epoch & 1
    uint8_t *out;
    AfskRxResult *res;
};

__device__ __forceinline__ long long num_windows(long long n, int bf, int clk)
{
    // K = #{k >= 0 : clk + k*bf < n - bf}   (afskmodem.py:362,372 — strict)
    const long long span = n - bf - clk;
    if (span <= 0) return 0;
    // captures of fewer than 2^31 samples (all but config-4-sized ones): a 32-bit division instead of the ~100 instructions
    // of a 64-bit one, which showed in the per-capture framing kernel
    if (span < (1ll << 31) - 4096) return (long long)(((uint32_t)span + (uint32_t)bf - 1u) / (uint32_t)bf);
    return (span + bf - 1) / bf;
}

// Waiting on another CTA of the same launch (fused schedule): a wait that has lasted four seconds is a scheduling
// bug, and an aborted launch (cudaErrorLaunchFailure at the next synchronisation) is better than a hung device.
__device__ __forceinline__ void spin_guard(unsigned long long &t0)
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    if (t0 == 0) t0 = t;
    else if (t - t0 > 4000000000ull) __trap();
}

// ------------------------------------------------------------------------------ k_clock ----
__global__ void __launch_bounds__(kClockThreads) k_clock(const int16_t *__restrict__ x,
                                                         const CapDesc *__restrict__ caps,
                                                         int32_t *__restrict__ clock,
                                                         AfskRxResult *__restrict__ res, uint32_t qmask)
{
    const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const CapDesc d = caps[c];
    if (d.status0 == 0 && (d.bf & 3) == 0 && d.bf <= 24 && ((qmask >> (d.bf >> 2)) & 1u)) return;   // k_clock_q's capture
    if (d.status0 != 0) {
        if (tid == 0) {
            clock[c] = -1;
            AfskRxResult r;
            r.status = d.status0; r.clock = -1; r.train_end = -1; r.nbits = 0; r.nbytes = 0;
            res[c] = r;
        }
        return;
    }
    // y = up to 4104 samples starting at the 16-byte boundary at or below the capture start.
    // Qs[4 + i] = y[0] + ... + y[i] (mod 2^32), Qs[3] = 0, so P[i] = sum y[0..i) = Qs[3 + i].
    __shared__ __align__(16) uint32_t Qs[4 + AFSK_SYNC_FRAMES + 8 + kClockThreads];
    __shared__ uint32_t warp_tot[kClockThreads / 32];
    __shared__ uint32_t warp_min[kClockThreads / 32];
    const uint32_t *P = Qs + 3;
    const int64_t ga = d.off & ~(int64_t)7;
    const int e = (int)(d.off - ga);
    const uint4 *src = reinterpret_cast<const uint4 *>(x + ga);
    // warp w scans samples [1024w, 1024w + 1024): 4 rounds of 32 coalesced 16-byte vectors
    uint32_t pre[4][8], vsum[4], voff[4];
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const uint4 qv = ld_nc_v4(src + warp * 128 + r * 32 + lane);
        const uint32_t wv[4] = {qv.x, qv.y, qv.z, qv.w};
        uint32_t run = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            run += (uint32_t)(int)(int16_t)(wv[j] & 0xFFFF); pre[r][2 * j] = run;
            run += (uint32_t)(int)(int16_t)(wv[j] >> 16);    pre[r][2 * j + 1] = run;
        }
        vsum[r] = run;
    }
    uint32_t carry = 0;
#pragma unroll
    for (int r = 0; r < 4; r++) {
        uint32_t inc = vsum[r];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
            if (lane >= o) inc += t;
        }
        voff[r] = carry + inc - vsum[r];
        carry += __shfl_sync(0xFFFFFFFFu, inc, 31);
    }
    if (lane == 0) warp_tot[warp] = carry;
    if (tid == 0) Qs[3] = 0;
    __syncthreads();
    uint32_t base = 0;
    for (int w = 0; w < warp; w++) base += warp_tot[w];
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const uint32_t o = base + voff[r];
        uint4 *dst = reinterpret_cast<uint4 *>(Qs + 4 + (warp * 128 + r * 32 + lane) * 8);
        dst[0] = make_uint4(o + pre[r][0], o + pre[r][1], o + pre[r][2], o + pre[r][3]);
        dst[1] = make_uint4(o + pre[r][4], o + pre[r][5], o + pre[r][6], o + pre[r][7]);
    }
    if (tid == kClockThreads - 1 && e > 0) {
        // an unaligned capture start needs the 513th vector (samples 4096..4103 of y)
        const uint4 qv = ld_nc_v4(src + 512);
        const uint32_t wv[4] = {qv.x, qv.y, qv.z, qv.w};
        uint32_t run = base + carry;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            run += (uint32_t)(int)(int16_t)(wv[j] & 0xFFFF); Qs[4 + 4096 + 2 * j] = run;
            run += (uint32_t)(int)(int16_t)(wv[j] >> 16);    Qs[4 + 4096 + 2 * j + 1] = run;
        }
    }
    __syncthreads();

    const int bf = d.bf, q = bf >> 2;
    const int span = AFSK_SYNC_FRAMES - 2 * bf;                 // :327
    const uint32_t c0 = 65535u * (uint32_t)bf;
    const uint32_t div = 2u * (uint32_t)bf;
    // getDiff(i) = floor(D_i / 2bf) is monotone in D_i, so the first strict minimum (:332-337) is the
    // first i with D_i <= T where T = (floor(min D / 2bf) + 1) * 2bf - 1: one division per capture.
    //
    // sum_j |T[j] - x[i+j]| over the training cycle (mark: q HI,q LO,q HI,q LO ; space: h HI,h LO) is
    //     D_i = c0 + t0 + t8 - 2 (t1 - t2 + t3 - t4 + t6),   t_m = P[i + m q]
    // and candidate i + q uses t1..t9: a thread walks a CHAIN i, i + q, i + 2q, ... with the nine taps in
    // registers and ONE new shared-memory word per candidate (instead of seven).  The candidates are
    // tiled in blocks of q * kClockChain; item (block b, residue a) is the chain starting at a + q * kClockChain * b,
    // so consecutive threads read consecutive words.  Every decodable baud from 300 up gives at most 128
    // items (one per thread); rarer geometries take further items through the direct seven-tap form.
    const uint32_t *Pe = P + e;
    const int qL = q * kClockChain;
    const int nitems = ((span + qL - 1) / qL) * q;
    auto D_at = [&](int i) -> uint32_t {
        return c0 + Pe[i] + Pe[i + 8 * q] - 2u * (Pe[i + q] - Pe[i + 2 * q] + Pe[i + 3 * q] - Pe[i + 4 * q] + Pe[i + 6 * q]);
    };
    uint32_t Dv[kClockChain];
    uint32_t best = 0xFFFFFFFFu;
    const int s0 = (tid % q) + qL * (tid / q);                  // first candidate of this thread's chain
    // kv valid candidates in the chain (a suffix may lie beyond the span, or the whole item may not exist);
    // a valid candidate reads P[.. 4103] at most, so loads guarded by k < kv stay inside Qs
    int kv = tid < nitems ? (span - s0 + q - 1) / q : 0;
    kv = kv < 0 ? 0 : (kv > kClockChain ? kClockChain : kv);
    {
        uint32_t t[9];
        uint32_t ta = afsk_smem_u32(P + (kv > 0 ? s0 + e : 0));
        const uint32_t tstep = 4u * (uint32_t)q;
#pragma unroll
        for (int m = 0; m < 8; m++) { t[m] = lds_u32(ta); ta += tstep; }
#pragma unroll
        for (int k = 0; k < kClockChain; k++) {
            t[8] = lds_u32_if(ta, k < kv);                      // undefined for k >= kv (never used)
            ta += tstep;
            const uint32_t D = c0 + t[0] + t[8] - 2u * (t[1] - t[2] + t[3] - t[4] + t[6]);
            Dv[k] = D;                                          // garbage for k >= kv: masked below
            if (k < kv) best = min(best, D);
#pragma unroll
            for (int m = 0; m < 8; m++) t[m] = t[m + 1];
        }
    }
    for (int it = tid + kClockThreads; it < nitems; it += kClockThreads) {
        const int s1 = (it % q) + qL * (it / q);
        for (int k = 0, i = s1; k < kClockChain && i < span; k++, i += q) best = min(best, D_at(i));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xFFFFFFFFu, best, o));
    if (lane == 0) warp_min[warp] = best;
    __syncthreads();
    best = warp_min[0];
#pragma unroll
    for (int w = 1; w < kClockThreads / 32; w++) best = min(best, warp_min[w]);
    const uint32_t T = (best / div + 1u) * div - 1u;            // getDiff :107
    uint32_t first = 0xFFFFFFFFu;
    {
        // smallest k with Dv[k] <= T; if that k is not a valid candidate, no valid one qualifies
        int kf = kClockChain;
#pragma unroll
        for (int k = kClockChain - 1; k >= 0; k--)
            if (Dv[k] <= T) kf = k;
        if (kf < kv) first = (uint32_t)(s0 + kf * q);
    }
    for (int it = tid + kClockThreads; it < nitems; it += kClockThreads) {
        const int s1 = (it % q) + qL * (it / q);
        for (int k = 0, i = s1; k < kClockChain && i < span; k++, i += q)
            if (D_at(i) <= T) { first = min(first, (uint32_t)i); break; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) first = min(first, __shfl_xor_sync(0xFFFFFFFFu, first, o));
    __syncthreads();
    if (lane == 0) warp_min[warp] = first;
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < kClockThreads / 32; w++) first = min(first, warp_min[w]);
        clock[c] = (int32_t)first;
    }
}

// ---------------------------------------------------------------------------- k_clock_q ----
// __recoverClockIndex (:322-339) for the short bits (bf = 4 Q, Q = 2..6: 6000 / 4000 / 3000 / 2400 / 2000 baud), where a
// batch holds the most captures per sample and k_clock's ~26 thread instructions per candidate show in the step.
// No prefix array, no shared memory, no shuffles: thread t scores the 32 candidates at positions 32 b .. 32 b + 31 of
// the 16-byte aligned sample stream y (b = the thread's block) from 4 + Q vectors it loads itself, all in registers:
//     a[j] = y[j] + ... + y[j + Q - 1]                      (IDP.2A with +/-1 byte selectors; sliding from Q = 4)
//     e[j] = a[j] - a[j + Q],   b[j] = a[j] + a[j + Q]
//     D_j  = c0 - (e[j] + e[j + 2Q]) - (b[j + 4Q] - b[j + 6Q])        sum |training cycle - y[j ..]|, c0 = 65535 bf
// (mark = +Q -Q +Q -Q, space = +2Q -2Q at full scale: |T - y| = 32767 - y or y + 32768), about 10 instructions per
// candidate.  getDiff = floor(D / 2bf) (:107) by one exact multiply-high (D < 2^22), and the first minimum (:332-337)
// is the minimum of the key (getDiff << 12) | position.  Candidate i sits at position i + e (e = capture start
// modulo 8 samples); positions outside [e, e + span) are masked.  They all lie in blocks 0, 126 and 127, which the
// block rotation b = (t + 126) & 127 puts into warp 0: the other three warps run the unmasked body.
template <int kQ>
__device__ __forceinline__ int clockq_sum(const uint32_t (&W)[16 + 4 * kQ], int j)
{
    // y[j] + ... + y[j + kQ - 1] straight from the words (samples 2k, 2k + 1 in W[k])
    int acc = 0;
#pragma unroll
    for (int k = j >> 1; k <= (j + kQ - 1) >> 1; k++) {
        const bool lo = 2 * k >= j, hi = 2 * k + 1 <= j + kQ - 1;
        acc = __dp2a_lo((int)W[k], (lo ? 0x0001 : 0) | (hi ? 0x0100 : 0), acc);
    }
    return acc;
}

template <int kQ, bool kMasked>
__device__ __forceinline__ uint32_t clockq_scan(const uint4 *__restrict__ src, int blk, int e, int span)
{
    constexpr int kNV = 4 + kQ, kNA = 32 + 7 * kQ, kNE = 32 + 2 * kQ;
    constexpr uint32_t kDiv = 8u * kQ;                                   // 2 bf
    constexpr uint32_t kMagic = (uint32_t)((0x100000000ull + kDiv - 1) / kDiv);   // floor(D / kDiv) == umulhi(D, kMagic), D < 2^22
    uint32_t W[4 * kNV];
#pragma unroll
    for (int r = 0; r < kNV; r++) {
        uint4 q = make_uint4(0u, 0u, 0u, 0u);
        const int v = 4 * blk + r;
        // the capture holds y[e, e + 4096): vectors 0..511, and vector 512 when its start is not aligned
        if (!kMasked || v < 512 || (v == 512 && e > 0)) q = ld_nc_v4(src + v);
        W[4 * r] = q.x; W[4 * r + 1] = q.y; W[4 * r + 2] = q.z; W[4 * r + 3] = q.w;
    }
    int a[kNA];
    if (kQ <= 3) {
#pragma unroll
        for (int j = 0; j < kNA; j++) a[j] = clockq_sum<kQ>(W, j);
    } else {
        a[0] = clockq_sum<kQ>(W, 0);
#pragma unroll
        for (int j = 0; j + 1 < kNA; j++) {
            const int t = __dp2a_lo((int)W[j >> 1], (j & 1) ? 0xFF00 : 0x00FF, a[j]);            // - y[j]
            a[j + 1] = __dp2a_lo((int)W[(j + kQ) >> 1], ((j + kQ) & 1) ? 0x0100 : 0x0001, t);   // + y[j + Q]
        }
    }
    int ee[kNE], bb[kNE];
#pragma unroll
    for (int j = 0; j < kNE; j++) {
        ee[j] = a[j] - a[j + kQ];
        bb[j] = a[j + 4 * kQ] + a[j + 5 * kQ];
    }
    const int c0 = 65535 * 4 * kQ;
    const int lo = e - 32 * blk, hi = e + span - 32 * blk;              // valid positions of the block: lo <= k < hi
    uint32_t best = 0xFFFFFFFFu;
#pragma unroll
    for (int k = 0; k < 32; k++) {
        const int f = c0 - bb[k] + bb[k + 2 * kQ];
        const uint32_t D = (uint32_t)(f - ee[k] - ee[k + 2 * kQ]);
        uint32_t key = __umulhi(D, kMagic) * 4096u + (uint32_t)(32 * blk + k);
        if (kMasked && (k < lo || k >= hi)) key = 0xFFFFFFFFu;
        best = min(best, key);
    }
    return best;
}

template <int kQ>
__global__ void __launch_bounds__(kClockThreads) k_clock_q(const int16_t *__restrict__ x, const CapDesc *__restrict__ caps,
                                                           const int32_t *__restrict__ gcaps, int32_t *__restrict__ clock)
{
    const int c = gcaps[blockIdx.x], tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t off = caps[c].off;
    const int64_t ga = off & ~(int64_t)7;
    const int e = (int)(off - ga);
    const uint4 *src = reinterpret_cast<const uint4 *>(x + ga);
    const int span = AFSK_SYNC_FRAMES - 8 * kQ;                          // :327
    const int blk = (tid + 126) & 127;
    __shared__ uint32_t warp_min[kClockThreads / 32];
    uint32_t best = warp == 0 ? clockq_scan<kQ, true>(src, blk, e, span) : clockq_scan<kQ, false>(src, blk, e, span);
    best = __reduce_min_sync(0xFFFFFFFFu, best);
    if (lane == 0) warp_min[warp] = best;
    __syncthreads();
    if (tid == 0) {
#pragma unroll
        for (int w = 1; w < kClockThreads / 32; w++) best = min(best, warp_min[w]);
        clock[c] = (int32_t)(best & 4095u) - e;
    }
}

// -------------------------------------------------------------------------- auxiliary warps ----
// Fused mode.  Every CTA of a demodulator launch carries two or four extra warps that never touch the sample
// ring.  Together (all CTAs) they work through two job lists of the launch's capture group, each handed out
// in capture order by a global counter:
//   clock jobs  __recoverClockIndex (:322-339) for one capture, by the CTA's auxiliary warps together;
//               the result is published as one 64-bit word {clock, epoch} that the producer warps poll
//               before they cut the capture into tiles.  Captures are needed in the same order as the jobs
//               are handed out, and a claimed job never blocks, so producers cannot starve.
//   frame jobs  the body of k_frame_warp for one capture, by one auxiliary warp, once every consumer warp of
//               every tile of the capture has arrived on the capture's counter (release / acquire).
// The arithmetic is the same as in k_clock / k_frame_warp; only the scheduling differs, so the three-kernel
// path stays as the reference the tests compare this one with (AFSK_OPT_FUSED).
// kAW auxiliary warps per CTA: 2 behind the general demodulator (its consumers need up to 77 registers, and
// two CTAs of 11 warps leave 88), 4 behind the short-window kernels (62-68 registers; their captures are the
// short ones, which need clock jobs at the highest rate)
constexpr int kAuxWarpsMax = 4;
constexpr int kFusedThreads2 = kDemodThreads + 64;
constexpr int kFusedThreads4 = kDemodThreads + 128;
constexpr int kAuxPass = 2048;                 // clock candidates per pass (the prefix array covers one pass)
constexpr int kAuxMaxVec = 304;                // 16-byte vectors of samples per pass: 2048 + 2 bf + 14 <= 2432
constexpr int kAuxMaxBf = (kAuxMaxVec * 8 - kAuxPass - 14) / 2;   // 185
constexpr int kAuxChain = 18;                  // candidates per chain (a quarter bit apart), see k_clock
constexpr int kAuxTileSlots = 64;              // tiles in flight between a CTA's consumer warps' reports (they are at most a ring apart)

struct __align__(16) AuxSmem {
    uint32_t Qs[4 + 8 * kAuxMaxVec];           // Qs[4 + i] = y[0] + ... + y[i], Qs[3] = 0 (as in k_clock)
    uint32_t warp_tot[kAuxWarpsMax];
    uint32_t warp_min[kAuxWarpsMax];
    int job[2];
    int q_pad0[2];
    uint32_t tile_arr[kAuxTileSlots];          // consumer warps that have reported tile n of this CTA, slot n % kAuxTileSlots
    uint8_t lut[128];
};

template <int kAW>
__device__ __forceinline__ void aux_bar()
{
    asm volatile("bar.sync 2, %0;" ::"n"(32 * kAW) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// plane words written by other CTAs of the same launch: read them from L2 (an L1 line could be stale)
__device__ __forceinline__ uint32_t ld_cg_u32(const uint32_t *p)
{
    uint32_t v;
    asm("ld.global.cg.u32 %0, [%1];" : "=r"(v) : "l"(p));    // not volatile: independent loads may be batched
    return v;
}

// Clock index of one capture by the 32 * kAW auxiliary threads of a CTA (atid = 0 .. 32 kAW - 1).
// Same closed form and chains as k_clock; differences: the 4096-frame window is scanned in passes of
// kAuxPass candidates so that the prefix array is 9.7 KB instead of 16.5 KB (the ring of the short-window
// kernels leaves no more), and the first minimum is found in ONE sweep as the minimum of the key
// (floor(D / 2bf) << 12) | i, the floor by a multiply-shift that is exact for D < 2^28.
template <int kAW>
__device__ uint32_t aux_clock_index(const int16_t *__restrict__ x, long long off, int bf, uint32_t magic, int shift,
                                    AuxSmem &S, int atid)
{
    constexpr int kAT = 32 * kAW;
    constexpr int kRounds = (kAuxMaxVec + kAT - 1) / kAT;       // vectors per thread and pass
    const int lane = atid & 31, warp = atid >> 5;
    const int q = bf >> 2, span = AFSK_SYNC_FRAMES - 2 * bf;    // :327
    const uint32_t c0 = 65535u * (uint32_t)bf;
    const int qL = q * kAuxChain;
    // item = chain (block b, residue a): candidates a + qL b, a + qL b + q, ...  (local to the pass)
    const int b_first = atid / q, a_first = atid - b_first * q;
    uint32_t best = 0xFFFFFFFFu;
    for (int s0 = 0; s0 < span; s0 += kAuxPass) {
        const int C = min(kAuxPass, span - s0);                 // candidates s0 .. s0 + C - 1
        const long long g0 = off + s0, ga = g0 & ~7LL;
        const int e = (int)(g0 - ga);
        const int nvec = (e + C + 2 * bf + 7) >> 3;             // <= kAuxMaxVec (bf <= kAuxMaxBf, checked on the host)
        const uint4 *src = reinterpret_cast<const uint4 *>(x + ga);
        // warp w scans vectors [w * VW, (w + 1) * VW): kRounds rounds of 32 coalesced 16-byte loads
        constexpr int VW = kRounds * 32;
        uint32_t carry = 0;
        uint32_t voff[kRounds];
        uint4 qv[kRounds];
#pragma unroll
        for (int r = 0; r < kRounds; r++) {
            const int v = warp * VW + r * 32 + lane;
            qv[r] = make_uint4(0u, 0u, 0u, 0u);
            if (v < nvec) qv[r] = ld_nc_v4(src + v);
        }
#pragma unroll
        for (int r = 0; r < kRounds; r++) {
            // sum of the vector's 8 samples: IDP.2A with weights (1, 1) adds both halves of a word
            int run = __dp2a_lo((int)qv[r].x, 0x0101, 0);
            run = __dp2a_lo((int)qv[r].y, 0x0101, run);
            run = __dp2a_lo((int)qv[r].z, 0x0101, run);
            run = __dp2a_lo((int)qv[r].w, 0x0101, run);
            uint32_t inc = (uint32_t)run;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
                if (lane >= o) inc += t;
            }
            voff[r] = carry + inc - (uint32_t)run;
            carry += __shfl_sync(0xFFFFFFFFu, inc, 31);
        }
        if (lane == 0) S.warp_tot[warp] = carry;
        if (atid == 0) S.Qs[3] = 0;
        aux_bar<kAW>();
        uint32_t base = 0;
        for (int w = 0; w < warp; w++) base += S.warp_tot[w];
#pragma unroll
        for (int r = 0; r < kRounds; r++) {
            const int v = warp * VW + r * 32 + lane;
            if (v < nvec) {
                const uint32_t wv[4] = {qv[r].x, qv[r].y, qv[r].z, qv[r].w};
                uint32_t run = base + voff[r], pre[8];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    run += (uint32_t)(int)(int16_t)(wv[j] & 0xFFFF); pre[2 * j] = run;
                    run += (uint32_t)(int)(int16_t)(wv[j] >> 16);    pre[2 * j + 1] = run;
                }
                uint4 *dst = reinterpret_cast<uint4 *>(S.Qs + 4 + v * 8);
                dst[0] = make_uint4(pre[0], pre[1], pre[2], pre[3]);
                dst[1] = make_uint4(pre[4], pre[5], pre[6], pre[7]);
            }
        }
        aux_bar<kAW>();
        // candidate s0 + il (il < C):  D = c0 + t0 + t8 - 2 (t1 - t2 + t3 - t4 + t6),  t_m = P[il + m q],
        // P[j] = Qs[3 + e + j]
        const uint32_t *Pe = S.Qs + 3 + e;
        int a = a_first, b = b_first;
        while (true) {
            const int st = a + qL * b;
            if (st >= C) break;                                  // blocks only grow from here
            uint32_t t[9];
            uint32_t ta = afsk_smem_u32(Pe + st);
            const uint32_t tstep = 4u * (uint32_t)q;
#pragma unroll
            for (int m = 0; m < 8; m++) { t[m] = lds_u32(ta); ta += tstep; }
            int il = st;
#pragma unroll
            for (int k = 0; k < kAuxChain; k++) {
                const bool valid = il < C;
                t[8] = lds_u32_if(ta, valid);                   // undefined past the pass (never used)
                ta += tstep;
                const uint32_t D = c0 + t[0] + t[8] - 2u * (t[1] - t[2] + t[3] - t[4] + t[6]);
                const uint32_t fl = (uint32_t)(((unsigned long long)D * magic) >> shift);     // getDiff :107
                const uint32_t key = (fl << 12) | (uint32_t)(s0 + il);
                if (valid) best = min(best, key);
                il += q;
#pragma unroll
                for (int m = 0; m < 8; m++) t[m] = t[m + 1];
            }
            // next item of this thread: it + kAT
            a += kAT % q; b += kAT / q;                          // kAT is a constant: one division by q per job
            if (a >= q) { a -= q; b++; }
        }
        aux_bar<kAW>();                                          // the next pass overwrites Qs
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xFFFFFFFFu, best, o));
    if (lane == 0) S.warp_min[warp] = best;
    aux_bar<kAW>();
    best = S.warp_min[0];
#pragma unroll
    for (int w = 1; w < kAW; w++) best = min(best, S.warp_min[w]);
    return best & 4095u;                                         // first index of the minimum (:332-337)
}

// k_clock2: the auxiliary warps' clock job (aux_clock_index) as a kernel of its own, one 128-thread CTA per capture.
// Against k_clock it needs 9.7 KB instead of 17 KB of shared memory and no 35-register array of candidate
// distances (one sweep with the key minimum), so more captures are in flight per SM; bit lengths up to kAuxMaxBf.
__global__ void __launch_bounds__(128, 12) k_clock2(const int16_t *__restrict__ x, const CapDesc *__restrict__ caps,
                                                int32_t *__restrict__ clock, AfskRxResult *__restrict__ res)
{
    __shared__ AuxSmem S;
    const int c = blockIdx.x, tid = threadIdx.x;
    const CapDesc d = caps[c];
    if (d.status0 != 0) {
        if (tid == 0) {
            clock[c] = -1;
            AfskRxResult r;
            r.status = d.status0; r.clock = -1; r.train_end = -1; r.nbits = 0; r.nbytes = 0;
            res[c] = r;
        }
        return;
    }
    const uint32_t dv = 2u * (uint32_t)d.bf;
    const int shift = 28 + (32 - __clz((int)(dv - 1u)));                 // 28 + ceil(log2 dv)
    const uint32_t magic = (uint32_t)((((unsigned long long)1 << shift) + dv - 1) / dv);
    const uint32_t clk = aux_clock_index<4>(x, d.off, d.bf, magic, shift, S, tid);
    if (tid == 0) clock[c] = (int32_t)clk;
}

// consumer-side state of fused framing (see signal_flush, defined with the framing code below): a consumer
// warp notes the capture of every tile it finishes, one tile per lane, and reports 32 of them at a time
struct TileSignal {
    int ci = -1;                 // this lane's noted tile: position of its capture in the group
    uint32_t want = 0;           // tiles that complete that capture
    int npend = 0;               // tiles noted since the last report (warp-uniform)
    int n0 = 0;                  // sequence number (in this CTA) of the first noted tile
    int seq = 0;                 // tiles seen so far
};
__device__ __forceinline__ void signal_flush(const DemodParams &p, AuxSmem &S, TileSignal &t, int lane);
__device__ __forceinline__ void signal_note(const DemodParams &p, AuxSmem &S, TileSignal &t, int ci, uint32_t want, int lane)
{
#ifdef AFSK_DBG_NOSIGNAL
    return;
#endif
    if (t.npend == 32) signal_flush(p, S, t, lane);   // the noted tiles' plane stores are at least one tile old
    if (t.npend == 0) t.n0 = t.seq;
    if (lane == t.npend) { t.ci = ci; t.want = want; }
    t.npend++;
    t.seq++;
}
__device__ __forceinline__ void signal_finish(const DemodParams &p, AuxSmem &S, TileSignal &t, int lane);
template <int kAW>
__device__ __forceinline__ void demod_aux(const DemodParams &p, uint8_t *smem);
// before the CTA's first barrier: the framing queue starts empty (the auxiliary threads exist only in fused mode)
__device__ __forceinline__ void aux_smem_init(const DemodParams &p, AuxSmem &S)
{
    if (!p.fused) return;
    const int atid = (int)threadIdx.x - kDemodThreads;
    if (atid < 0) return;
    for (int i = atid; i < kAuxTileSlots; i += 64) S.tile_arr[i] = 0u;
}

// ------------------------------------------------------------------------------ k_demod ----
// Per-sample classification (Receiver.__amplify :287-296) and the two getDiff sums (:346-347)
// in packed integer form.  For a sample x let p = [x > 512], n = [x < -512], c = p - n.
// With T the +/-1 template (mark: + - + - per quarter, space: + + - -):
//     sum_j |T[j] - amp[j]| = (65535 * (bf - T.c) + T.(p+n)) / 2          (DESIGN.md §3)
// so each window needs U = T.c and Xn = T.n for both templates plus A = sum |x|.
//
// Four samples (two 32-bit words) per step:
//   g  = min((x + 512) mod 2^16, 1025)   VIADDMNMX.U16x2    g == 1025  <=>  |x| > 512
//   t  = g + 0x7BFF                      bit 15 of each half <=> |x| > 512
//   S4 / NZ4 = sign / non-zero byte masks of the 4 samples (PRMT with sign replication)
//   v4 = NZ4 & (S4 | 1)                  bytes: 1 (x > 512), 255 (x < -512), 0
//   acc += dp4a.u32.s32(v4, T4)          = 256 * T.n + T.c   (IDP.4A; decoded per <= 120 samples)
//   A   += dp2a.s16.s8(x, (S4 | 1) & inwindow)  = sum sign(x) * x      (IDP.2A)
__device__ __forceinline__ int dp4a_us(uint32_t a, uint32_t b, int c)
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

__device__ __forceinline__ void accum4(uint32_t w0, uint32_t w1, uint32_t mw, uint32_t sw, uint32_t aw, uint32_t k512,
                                       int &accM, int &accS, int &accA)
{
    const uint32_t g0 = __viaddmin_u16x2(w0, k512, 0x04010401u);
    const uint32_t g1 = __viaddmin_u16x2(w1, k512, 0x04010401u);
    const uint32_t t0 = g0 + 0x7BFF7BFFu;
    const uint32_t t1 = g1 + 0x7BFF7BFFu;
    const uint32_t s4 = prmt(w0, w1, 0xFDB9u);            // 0xFF where x < 0
    const uint32_t nz4 = prmt(t0, t1, 0xFDB9u);           // 0xFF where |x| > 512
    const uint32_t v4 = nz4 & (s4 | 0x01010101u);
    const uint32_t sg4 = (s4 | 0x01010101u) & aw;         // +1 / -1 inside the window, 0 outside
    accM = dp4a_us(v4, mw, accM);
    accS = dp4a_us(v4, sw, accS);
    accA = __dp2a_lo((int)w0, (int)sg4, accA);
    accA = __dp2a_hi((int)w1, (int)sg4, accA);
}

// acc = 256 * Xn + U with |U| <= 127
__device__ __forceinline__ void unpack_acc(int acc, int &U, int &Xn)
{
    const int u = (int)((unsigned)acc << 24) >> 24;
    U += u;
    Xn += (acc - u) >> 8;
}

// The bit of a window whose correlations tie (Um == Us) while Ns > Nm: mark_diff < space_diff (:346-351) compares
// floor(M / bf) < floor(S / bf), with 2 M = 65535 bf - 65534 Um + 2 Nm and 2 S = 2 M + 2 (Ns - Nm)
__device__ __forceinline__ bool tie_bit(int Um, int Nm, int Ns, int bf)
{
    const int two_bf = 2 * bf;
    const int M2 = 65535 * bf - 65534 * Um + 2 * Nm;
    const int S2 = M2 + 2 * (Ns - Nm);
    return (S2 - M2 >= two_bf) || (M2 < (S2 / two_bf) * two_bf);
}

// accum4 with every slot inside the window
__device__ __forceinline__ void accum4_full(uint32_t w0, uint32_t w1, uint32_t mw, uint32_t sw, uint32_t k512,
                                            int &accM, int &accS, int &accA)
{
    const uint32_t g0 = __viaddmin_u16x2(w0, k512, 0x04010401u);
    const uint32_t g1 = __viaddmin_u16x2(w1, k512, 0x04010401u);
    const uint32_t t0 = g0 + 0x7BFF7BFFu;
    const uint32_t t1 = g1 + 0x7BFF7BFFu;
    const uint32_t s4 = prmt(w0, w1, 0xFDB9u);
    const uint32_t nz4 = prmt(t0, t1, 0xFDB9u);
    const uint32_t sg4 = s4 | 0x01010101u;
    const uint32_t v4 = nz4 & sg4;
    accM = dp4a_us(v4, mw, accM);
    accS = dp4a_us(v4, sw, accS);
    accA = __dp2a_lo((int)w0, (int)sg4, accA);
    accA = __dp2a_hi((int)w1, (int)sg4, accA);
}

// Fast path of the merge-mode kernel.  mark - space = 2 D with D = (0, -1, +1, 0) per quarter, so
//     acc += dp4a.u32.s32(v4, D4)   = 256 * D.n + D.c ,   D.c = (Um - Us) / 2 ,  D.n = (Nm - Ns) / 2
// decides the bit whenever Um != Us or Ns <= Nm (see the decision below); one IDP.4A instead of two.
__device__ __forceinline__ void accum4_d(uint32_t w0, uint32_t w1, uint32_t dw, uint32_t k512, int &accD, int &accA)
{
    const uint32_t g0 = __viaddmin_u16x2(w0, k512, 0x04010401u);
    const uint32_t g1 = __viaddmin_u16x2(w1, k512, 0x04010401u);
    const uint32_t t0 = g0 + 0x7BFF7BFFu;
    const uint32_t t1 = g1 + 0x7BFF7BFFu;
    const uint32_t s4 = prmt(w0, w1, 0xFDB9u);
    const uint32_t nz4 = prmt(t0, t1, 0xFDB9u);
    const uint32_t sg4 = s4 | 0x01010101u;
    accD = dp4a_us(nz4 & sg4, dw, accD);
    accA = __dp2a_lo((int)w0, (int)sg4, accA);
    accA = __dp2a_hi((int)w1, (int)sg4, accA);
}
// amplitude only: four samples whose D weights are all zero
__device__ __forceinline__ void accum4_a(uint32_t w0, uint32_t w1, int &accA)
{
    const uint32_t sg4 = prmt(w0, w1, 0xFDB9u) | 0x01010101u;
    accA = __dp2a_lo((int)w0, (int)sg4, accA);
    accA = __dp2a_hi((int)w1, (int)sg4, accA);
}

// keep every 2nd / 4th bit of a ballot, packed to the low 16 / 8 bits
__device__ __forceinline__ uint32_t squeeze2(uint32_t x)
{
    x &= 0x55555555u;
    x = (x | (x >> 1)) & 0x33333333u;
    x = (x | (x >> 2)) & 0x0F0F0F0Fu;
    x = (x | (x >> 4)) & 0x00FF00FFu;
    return (x | (x >> 8)) & 0xFFFFu;
}
__device__ __forceinline__ uint32_t squeeze4(uint32_t x)
{
    x &= 0x11111111u;
    x = (x | (x >> 3)) & 0x03030303u;
    x = (x | (x >> 6)) & 0x000F000Fu;
    return (x | (x >> 12)) & 0xFFu;
}

constexpr int kFlushVecs = 15;      // 120 samples: keeps |T.c| <= 127 inside one packed accumulator

// Tiles are dealt round-robin: CTA b handles tiles b, b + G, b + 2G, ... (balanced to one tile; at any
// moment the whole grid streams one contiguous span of the sample buffer).  The producer WARP prepares tiles 32 at a time: lane j resolves tile
// n + j (tile -> capture map, capture descriptor, clock index: three dependent global loads) one
// batch ahead of use, then the lanes take turns feeding the shared-memory ring: tile metadata,
// mbarrier expect_tx, one 1-D TMA bulk copy per tile.
struct TileJob {
    TileMeta m;
    long long ga;        // first sample of the bulk copy
    uint32_t bytes;      // 0: no valid window in the tile
};

__device__ __forceinline__ TileJob demod_tile_job(const DemodParams &p, int it, long long base_mis)
{
    TileJob j;
    const int ci = p.tile_gpos[it];
    const int c = p.gcaps[ci];
    const int first = p.gtile_first[ci];
    const int4 d0 = *reinterpret_cast<const int4 *>(&p.caps[c].off);          // off, n
    const int4 d1 = *reinterpret_cast<const int4 *>(&p.caps[c].plane_base);   // plane_base, out_off
    const int thr = p.caps[c].thr;
    int clk;
    if (p.fused) {
        // the capture's clock job was handed out before any job of a later capture and never blocks
        unsigned long long w = ld_relaxed_u64(p.cready + c);
        unsigned long long t0 = 0;
        while ((uint32_t)(w >> 32) != p.epoch) { __nanosleep(200); spin_guard(t0); w = ld_relaxed_u64(p.cready + c); }
        clk = (int)(uint32_t)w;
    } else {
        clk = p.clock[c];
    }
    const long long off = ((long long)d0.y << 32) | (unsigned)d0.x, n = ((long long)d0.w << 32) | (unsigned)d0.z;
    const long long plane_base = ((long long)d1.y << 32) | (unsigned)d1.x;
    const long long K = num_windows(n, p.bf, clk);
    const long long k0t = (long long)(it - first) * p.wt;
    const long long nw = K - k0t;
    const int nwin = nw <= 0 ? 0 : (nw > p.wt ? p.wt : (int)nw);
    const long long g0 = off + clk + k0t * p.bf;             // first sample of the tile
    // copy from the 128-byte line holding that sample (misaligned bulk copies cost ~3.5 % of the
    // read bandwidth), unless the line starts before the buffer
    long long ga = ((g0 + base_mis) & ~63LL) - base_mis;
    if (ga < 0) ga = g0 & ~7LL;
    j.m.e0 = (int)(g0 - ga);
    j.m.nwin = nwin;
    j.m.thr_bf = thr * p.bf;
    j.m.gpos = ci;
    j.m.word_base = plane_base + (k0t >> 5);
    j.m.want = (uint32_t)(p.gtile_first[ci + 1] - first);
    j.m.pad2 = 0;
    j.ga = ga;
    j.bytes = nwin > 0 ? (uint32_t)((((long long)j.m.e0 + (long long)nwin * p.bf) * 2 + 15) & ~15LL) : 0u;
    return j;
}

__device__ __forceinline__ void demod_produce(const DemodParams &p, int ntile, uint8_t *stage_base, TileMeta *meta,
                                              uint64_t *full, uint64_t *empty)
{
    const int S = p.stages, lane = threadIdx.x & 31;
    const int G = (int)gridDim.x, first_tile = (int)blockIdx.x;
    const long long base_mis = (long long)((reinterpret_cast<uintptr_t>(p.samples) >> 1) & 63);   // multiple of 8
    int s = 0;
    uint32_t ph = 0;                                       // parity of the use count of stage s
    const uint64_t pol = l2_policy_evict_first();
    const bool hint = p.l2_hint != 0;
    // Tile jobs are resolved a batch ahead of their use, 32 at a time.  In fused mode a job waits for its
    // capture's clock, and at the start of the launch only one clock job per CTA can be under way: the first
    // two batches are 8 tiles, so that the stream starts after the first round of clock jobs.
    int bs = p.fused ? 8 : 32;
    TileJob next = {};
    if (lane < bs && lane < ntile) next = demod_tile_job(p, first_tile + lane * G, base_mis);
    for (int base = 0; base < ntile;) {
        const TileJob cur = next;
        const int nbs = (p.fused && base + bs < 16) ? 8 : 32;      // size of the batch after this one
        if (lane < nbs && base + bs + lane < ntile) next = demod_tile_job(p, first_tile + (base + bs + lane) * G, base_mis);
        const int cnt = min(bs, ntile - base);
        for (int j = 0; j < cnt; j++) {
            if (lane == j) {
                if (base + j >= S) {
                    while (!mbar_try_wait(&empty[s], ph ^ 1u)) __nanosleep(128);
                }
                meta[s] = cur.m;
                if (cur.bytes) {
                    mbar_arrive_expect_tx(&full[s], cur.bytes);
                    if (hint) bulk_g2s_hint(stage_base + (size_t)s * p.stage_bytes, p.samples + cur.ga, cur.bytes, &full[s], pol);
                    else bulk_g2s(stage_base + (size_t)s * p.stage_bytes, p.samples + cur.ga, cur.bytes, &full[s]);
                } else {
                    mbar_arrive(&full[s]);
                }
            }
            // the lanes must feed the ring in tile order: a lane two uses of a stage ahead would see
            // the parity it waits for already satisfied by the previous use
            __syncwarp();
            if (++s == S) { s = 0; ph ^= 1u; }
        }
        base += bs;
        bs = nbs;
    }
}

// Producer of the padded layout (k_demod_shift<.., kPad = true>: thread segments of 2^k vectors, 1500 / 750 / 375 baud).
// A thread per window would read 16-byte vectors 64 / 128 / 256 bytes apart: 4- to 8-way bank conflicts however the
// windows are dealt.  Here the tile is laid out with ONE spare vector after every thread segment of kV vectors (stride
// kV + 1: odd, conflict-free), which a bulk copy cannot do: the producer warp issues 16-byte cp.async copies (LDGSTS,
// 512 consecutive bytes per instruction) with the destination vector v + (v - v0) / kV, v0 = vector of the tile's first
// sample.  Each lane reports its copies to the stage's full barrier (cp.async.mbarrier.arrive.noinc), the lane that
// wrote the tile's metadata adds a plain arrival: 33 arrivals per use.
template <int kV>
__device__ __forceinline__ void demod_produce_pad(const DemodParams &p, int ntile, uint8_t *stage_base, TileMeta *meta,
                                                  uint64_t *full, uint64_t *empty, int pw, int npw)
{
    const int S = p.stages, lane = threadIdx.x & 31;
    const int G = (int)gridDim.x, first_tile = (int)blockIdx.x;
    const long long base_mis = (long long)((reinterpret_cast<uintptr_t>(p.samples) >> 1) & 63);
    int s = 0;
    uint32_t ph = 0;
    const uint64_t pol = l2_policy_evict_first();
    const bool hint = p.l2_hint != 0;
    const int vstep = 32 * npw, stage_bytes = p.stage_bytes;
    const uint32_t sdst = afsk_smem_u32(stage_base);
    const int16_t *samples = p.samples;
    TileJob next = {};
    if (lane < ntile) next = demod_tile_job(p, first_tile + lane * G, base_mis);
    for (int base = 0; base < ntile; base += 32) {
        const TileJob cur = next;
        if (base + 32 + lane < ntile) next = demod_tile_job(p, first_tile + (base + 32 + lane) * G, base_mis);
        const int cnt = min(32, ntile - base);
        for (int j = 0; j < cnt; j++) {
            const long long ga = __shfl_sync(0xFFFFFFFFu, cur.ga, j);
            const int nvec = (int)(__shfl_sync(0xFFFFFFFFu, cur.bytes, j) >> 4);
            const int v0 = __shfl_sync(0xFFFFFFFFu, cur.m.e0, j) >> 3;
            if (base + j >= S) {
                if (lane == 0)
                    while (!mbar_try_wait(&empty[s], ph ^ 1u)) __nanosleep(64);
                __syncwarp();
            }
            if (lane == j && pw == 0) {
                meta[s] = cur.m;
                mbar_arrive(&full[s]);
            }
            // vector v0 + u of the copy goes to vector v0 + u + u / kV of the stage; this lane: u = 32 pw + lane + k vstep
            const int nu = nvec - v0;
            int u = 32 * pw + lane;
            uint32_t d = sdst + (uint32_t)s * (uint32_t)stage_bytes + 16u * (uint32_t)(v0 + u);
            const char *sp = reinterpret_cast<const char *>(samples + ga) + 16 * (v0 + u);
            if (hint) {
                for (; u + 3 * vstep < nu; u += 4 * vstep, d += 64u * vstep, sp += 64 * vstep) {
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        cp_async16_hint(d + 16u * (uint32_t)(k * vstep) + 16u * ((uint32_t)(u + k * vstep) / (uint32_t)kV), sp + 16 * k * vstep, pol);
                }
                for (; u < nu; u += vstep, d += 16u * vstep, sp += 16 * vstep) cp_async16_hint(d + 16u * ((uint32_t)u / (uint32_t)kV), sp, pol);
            } else {
                for (; u + 3 * vstep < nu; u += 4 * vstep, d += 64u * vstep, sp += 64 * vstep) {
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        cp_async16(d + 16u * (uint32_t)(k * vstep) + 16u * ((uint32_t)(u + k * vstep) / (uint32_t)kV), sp + 16 * k * vstep);
                }
                for (; u < nu; u += vstep, d += 16u * vstep, sp += 16 * vstep) cp_async16(d + 16u * ((uint32_t)u / (uint32_t)kV), sp);
            }
            cp_async_mbar_arrive_noinc(&full[s]);
            if (++s == S) { s = 0; ph ^= 1u; }
        }
    }
}

// kNT > 0: the number of vector steps per thread is a compile-time constant (fully unrolled, one
// packed accumulator); kNT == 0: run-time count with a flush every kFlushVecs vectors.
// kMerge: the thread segment is a multiple of 8 samples, so the partial head vector (slots >= e)
// and the partial tail vector (slots < e) are merged into one full vector with 4 PRMTs.
template <int kNT, bool kMerge>
__global__ void __launch_bounds__(kFusedThreads2, 2) k_demod(const DemodParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int S = p.stages;
    const int tpw = 1 << p.tpw_log2;
    uint8_t *stage_base = smem;
    uint4 *wtab = reinterpret_cast<uint4 *>(smem + (size_t)S * p.stage_bytes);
    // entry (part, e, i) = two uint4 at wtab[part * PSq + e * ESq + 2 * i]; the odd strides put the
    // entries that the lanes of one warp read together (different part / e) in different banks
    const int wtab_entries = tpw * 8 * p.nt;
    const int ESq = 2 * p.nt + 1, PSq = 8 * ESq + 1;
    TileMeta *meta = reinterpret_cast<TileMeta *>(wtab + tpw * PSq);
    uint64_t *full = reinterpret_cast<uint64_t *>(meta + kMaxStages);
    uint64_t *empty = full + kMaxStages;
    uint8_t *resbuf = reinterpret_cast<uint8_t *>(empty + kMaxStages);   // [2][kConsumerThreads]

    // ---- template weight table: entry (part, e, i), slot s = 0..7 of vector i covers segment
    //      sample r = 8i + s - e (merge mode, i == 0: slots below e come from the tail vector,
    //      r = 8*nt + s - e); window position pos = part*seg + r; quarter pos/q gives the sign.
    //      Layout: {mark[0..3], mark[4..7], space[0..3], space[4..7]} {inwin[0..3], inwin[4..7], selA, selB}
    //      selA/selB: PRMT selectors (16 bits each) building the merged vector from head/tail words.
    {
        const int q = p.bf >> 2;
        for (int idx = tid; idx < wtab_entries; idx += (int)blockDim.x) {
            const int i = idx % p.nt, e = (idx / p.nt) & 7, part = idx / (p.nt * 8);
            const int seg_lo = part * p.seg, seg_hi = min(p.bf, seg_lo + p.seg);
            uint32_t mk[2] = {0u, 0u}, sp[2] = {0u, 0u}, in[2] = {0u, 0u}, sel[2] = {0u, 0u};
#pragma unroll
            for (int s = 0; s < 8; s++) {
                int r = 8 * i + s - e;
                if (kMerge && i == 0 && s < e) r += 8 * p.nt;
                const int pos = seg_lo + r;
                if (r >= 0 && pos < seg_hi) {
                    const int qd = pos / q;
                    const int sh = 8 * (s & 3);
                    mk[s >> 2] |= ((qd & 1) ? 0xFFu : 0x01u) << sh;    // mark : + - + -
                    sp[s >> 2] |= ((qd & 2) ? 0xFFu : 0x01u) << sh;    // space: + + - -
                    in[s >> 2] |= 0xFFu << sh;
                }
            }
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint32_t sj = (2 * j >= e) ? 0x3210u : ((2 * j + 1 < e) ? 0x7654u : 0x3254u);
                sel[j >> 1] |= sj << (16 * (j & 1));
            }
            uint4 *ent = wtab + part * PSq + e * ESq + 2 * i;
            ent[0] = make_uint4(mk[0], mk[1], sp[0], sp[1]);
            if (kMerge) {
                // every slot is inside the window; keep D = (mark - space) / 2 in place of the masks:
                // bytes differ (0x01 ^ 0xFF = 0xFE) exactly where D = mark
                const uint32_t x0 = mk[0] ^ sp[0], x1 = mk[1] ^ sp[1];
                in[0] = mk[0] & prmt(x0, x0, 0xBA98u);
                in[1] = mk[1] & prmt(x1, x1, 0xBA98u);
            }
            ent[1] = make_uint4(in[0], in[1], sel[0], sel[1]);
        }
    }
    if (tid == 0) {
        for (int s = 0; s < S; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kConsumerThreads / 32);
        }
        mbar_fence_init();
    }
    AuxSmem &AS = *reinterpret_cast<AuxSmem *>(smem + p.aux_off);
    aux_smem_init(p, AS);
    __syncthreads();

    const int ntile = (p.total_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles b, b + G, ...
    if (ntile <= 0) return;                          // never in fused mode: the grid is at most one CTA per tile

    if (warp == kConsumerThreads / 32) {
        demod_produce(p, ntile, stage_base, meta, full, empty);
        return;
    }
    if (warp > kConsumerThreads / 32) {
        demod_aux<2>(p, smem);
        return;
    }
    TileSignal sig;

    // ---------------------------------------------------------------- consumers ----
    const int w = tid >> p.tpw_log2, part = tid & (tpw - 1);
    const int wsub = kConsumerThreads >> p.tpw_log2;          // windows per sub-tile
    const int bf = p.bf, nv = p.nv;
    const int rel0 = w * bf + part * p.seg;
    // VIADDMNMX takes one immediate; derive the other constant from a runtime value so that it
    // lives in one register instead of being re-materialised before every use (stages < 65536)
    const uint32_t k512 = 0x02000200u | ((uint32_t)p.stages >> 16);
    // merge-mode fast path: D weights and head/tail selectors of the current alignment (registers)
    uint32_t Dw[kNT > 0 ? kNT : 1][2], selA = 0, selB = 0;
    int cur_al = -1;
    const bool v0_quarter03 = kMerge && kNT >= 4 && p.tpw_log2 == 0;
    constexpr bool kRot = kMerge && kNT == 4;                 // only 32-sample segments have four whole vectors
    const int rot = (kRot && p.rot) ? ((tid >> 1) & 3) : 0;
    int s = 0;
    uint32_t ph = 0;
    for (int n = 0; n < ntile; ++n) {
        mbar_wait(&full[s], ph);
        const TileMeta m = meta[s];
        if (p.fused_frame) signal_note(p, AS, sig, m.gpos, m.want, lane);
        // a tile is nsub sub-tiles of kConsumerThreads >> tpw_log2 windows each: where a thread's segment is short
        // (16 samples at 1500 / 750 / 375 baud, so that 128-bit loads are 2-way instead of 4-way bank conflicted) the
        // tile still is 32 KB, which is what the copy engine wants (8 KB tiles: 4.7 TB/s, 32 KB: 6.7)
#pragma unroll 1
        for (int u = 0; u < p.nsub; u++) {
        const int wbase = u * wsub;                            // first window of the sub-tile
        bool bit = false, quiet = false;
        if (m.nwin > wbase) {
            const int rel = m.e0 + rel0 + wbase * bf;
            const uint4 *dp = reinterpret_cast<const uint4 *>(stage_base + (size_t)s * p.stage_bytes) + (rel >> 3);
            const uint4 *wp = wtab + part * PSq + (rel & 7) * ESq;
            int Um = 0, Nm = 0, Us = 0, Ns = 0, accA = 0;
            bool b1;
            if (kMerge) {
                // ---- fast path: one packed accumulator of D = (mark - space) / 2 ----
                // bf % 8 == 0 here, so every window of the tile has the alignment m.e0 & 7 and a thread's
                // weights change only when the capture does: they are cached in registers
                // kRot (32-sample segments, 64 bytes between threads: a 128-bit load of the same vector index by a quarter
                // warp is a 4-way bank conflict): thread t takes its four vectors in the order (i + (t >> 1)) & 3, which
                // spreads the eight threads over all banks.  The sums do not care about the order; the weights are cached
                // in the same rotated order, and the head / tail merge of logical vector 0 becomes a PRMT with identity
                // selectors for the other three.
                if ((m.e0 & 7) != cur_al) {
                    cur_al = m.e0 & 7;
#pragma unroll
                    for (int i = 0; i < kNT; i++) {
                        const int li = kRot ? ((i + rot) & 3) : i;      // rot == 0 when the rotation is switched off
                        const uint4 av = wp[2 * li + 1];
                        Dw[i][0] = av.x; Dw[i][1] = av.y;
                    }
                    const uint4 a0 = wp[1];
                    selA = a0.z; selB = a0.w;
                }
                int accD = 0;
#pragma unroll
                for (int i = 0; i < kNT; i++) {
                    if (kRot && p.rot) {
                        const int li = (i + rot) & 3;
                        const bool head = li == 0;
                        uint4 dv = dp[li];
                        const uint4 tv = head ? dp[kNT] : dv;      // tail vector: slots below e (logical vector 0 only)
                        const uint32_t sA = head ? selA : 0x32103210u, sB = head ? selB : 0x32103210u;
                        dv.x = prmt(dv.x, tv.x, sA);
                        dv.y = prmt(dv.y, tv.y, sA >> 16);
                        dv.z = prmt(dv.z, tv.z, sB);
                        dv.w = prmt(dv.w, tv.w, sB >> 16);
                        accum4_d(dv.x, dv.y, Dw[i][0], k512, accD, accA);
                        accum4_d(dv.z, dv.w, Dw[i][1], k512, accD, accA);
                        continue;
                    }
                    uint4 dv = dp[i];
                    if (i == 0) {
                        const uint4 tv = dp[kNT];                  // tail vector: slots below e
                        dv.x = prmt(dv.x, tv.x, selA);
                        dv.y = prmt(dv.y, tv.y, selA >> 16);
                        dv.z = prmt(dv.z, tv.z, selB);
                        dv.w = prmt(dv.w, tv.w, selB >> 16);
                    }
                    if (i == 0 && v0_quarter03) {
                        // one thread per window, quarters of >= 8 samples: the merged vector lies in the
                        // last and first quarter, where mark and space agree (D == 0)
                        accum4_a(dv.x, dv.y, accA);
                        accum4_a(dv.z, dv.w, accA);
                    } else {
                        accum4_d(dv.x, dv.y, Dw[i][0], k512, accD, accA);
                        accum4_d(dv.z, dv.w, Dw[i][1], k512, accD, accA);
                    }
                }
                int dh = (int)((unsigned)accD << 24) >> 24;          // (Um - Us) / 2
                int nh = (accD - dh) >> 8;                           // (Nm - Ns) / 2
                for (int o = 1; o < tpw; o <<= 1) {
                    dh += __shfl_xor_sync(0xFFFFFFFFu, dh, o);
                    nh += __shfl_xor_sync(0xFFFFFFFFu, nh, o);
                    accA += __shfl_xor_sync(0xFFFFFFFFu, accA, o);
                }
                // 2 * (S - M) = 65534 * (Um - Us) + 2 * (Ns - Nm) with |Ns - Nm| <= bf: the sign of
                // Um - Us decides; on a tie S <= M (bit 0) unless Ns > Nm, and only then are the two
                // floors compared, which needs the full sums (rare: noise-only windows)
                b1 = dh > 0;
                if (__any_sync(0xFFFFFFFFu, dh == 0 && nh < 0)) {
                    int accM = 0, accS = 0, accA2 = 0;
#pragma unroll
                    for (int i = 0; i < kNT; i++) {
                        uint4 dv = dp[i];
                        const uint4 wv = wp[2 * i];
                        if (i == 0) {
                            const uint4 tv = dp[kNT];
                            dv.x = prmt(dv.x, tv.x, selA);
                            dv.y = prmt(dv.y, tv.y, selA >> 16);
                            dv.z = prmt(dv.z, tv.z, selB);
                            dv.w = prmt(dv.w, tv.w, selB >> 16);
                        }
                        accum4_full(dv.x, dv.y, wv.x, wv.z, k512, accM, accS, accA2);
                        accum4_full(dv.z, dv.w, wv.y, wv.w, k512, accM, accS, accA2);
                    }
                    unpack_acc(accM, Um, Nm);
                    unpack_acc(accS, Us, Ns);
                    for (int o = 1; o < tpw; o <<= 1) {
                        Um += __shfl_xor_sync(0xFFFFFFFFu, Um, o);
                        Nm += __shfl_xor_sync(0xFFFFFFFFu, Nm, o);
                        Us += __shfl_xor_sync(0xFFFFFFFFu, Us, o);
                        Ns += __shfl_xor_sync(0xFFFFFFFFu, Ns, o);
                    }
                    if (Um == Us && Ns > Nm) b1 = tie_bit(Um, Nm, Ns, bf);
                }
            } else {
                if (kNT > 0) {
                    int accM = 0, accS = 0;
#pragma unroll
                    for (int i = 0; i < kNT; i++) {
                        const uint4 dv = dp[i];
                        const uint4 wv = wp[2 * i];
                        const uint4 av = wp[2 * i + 1];
                        accum4(dv.x, dv.y, wv.x, wv.z, av.x, k512, accM, accS, accA);
                        accum4(dv.z, dv.w, wv.y, wv.w, av.y, k512, accM, accS, accA);
                    }
                    unpack_acc(accM, Um, Nm);
                    unpack_acc(accS, Us, Ns);
                } else {
                    for (int i0 = 0; i0 < nv; i0 += kFlushVecs) {
                        const int i1 = min(nv, i0 + kFlushVecs);
                        int accM = 0, accS = 0;
                        for (int i = i0; i < i1; i++) {
                            const uint4 dv = dp[i];
                            const uint4 wv = wp[2 * i];
                            const uint2 av = *reinterpret_cast<const uint2 *>(wp + 2 * i + 1);
                            accum4(dv.x, dv.y, wv.x, wv.z, av.x, k512, accM, accS, accA);
                            accum4(dv.z, dv.w, wv.y, wv.w, av.y, k512, accM, accS, accA);
                        }
                        unpack_acc(accM, Um, Nm);
                        unpack_acc(accS, Us, Ns);
                    }
                }
                for (int o = 1; o < tpw; o <<= 1) {
                    Um += __shfl_xor_sync(0xFFFFFFFFu, Um, o);
                    Nm += __shfl_xor_sync(0xFFFFFFFFu, Nm, o);
                    Us += __shfl_xor_sync(0xFFFFFFFFu, Us, o);
                    Ns += __shfl_xor_sync(0xFFFFFFFFu, Ns, o);
                    accA += __shfl_xor_sync(0xFFFFFFFFu, accA, o);
                }
                // 2 * sum|T - amp| = 65535 * bf - 65534 * U + 2 * Xn       (mark_diff < space_diff :346-351)
                // so 2 * (S - M) = 65534 * (Um - Us) + 2 * (Ns - Nm) with |Ns - Nm| <= bf: the sign of
                // Um - Us decides unless the correlations tie, and only then is the floor compared.
                const int du = Um - Us;
                b1 = du > 0;
                if (du == 0 && Ns > Nm) b1 = tie_bit(Um, Nm, Ns, bf);
            }
            const bool valid = (part == 0) && (wbase + w < m.nwin);
            bit = valid && b1;
            quiet = valid && (accA < m.thr_bf);                // getAmplitude(chunk) < amp_end :375
        }
        if (u == p.nsub - 1) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);               // stage may be refilled
        }
        if (m.nwin > wbase) {
            const long long word0 = m.word_base + (wbase >> 5);
            const int nleft = m.nwin - wbase;                    // valid windows from this sub-tile on
            if (p.tpw_log2 == 0) {
                const uint32_t bw = __ballot_sync(0xFFFFFFFFu, bit);
                const uint32_t qw = __ballot_sync(0xFFFFFFFFu, quiet);
                if (lane == 0 && warp * 32 < nleft) p.planes[word0 + warp] = make_uint2(bw, qw);
            } else if (p.tpw_log2 <= 2) {
                // 2 or 4 threads per window: the part-0 lanes hold the decisions; squeeze the
                // stride-tpw ballot into 16 / 8 bits and store them as a sub-word of the plane
                // (no CTA-wide barrier on this path)
                uint32_t bw = __ballot_sync(0xFFFFFFFFu, bit);
                uint32_t qw = __ballot_sync(0xFFFFFFFFu, quiet);
                const int per_warp = 32 >> p.tpw_log2;
                const int w0 = warp * per_warp;
                if (lane == 0 && (w0 & ~31) < nleft) {           // every piece of a word that holds a valid window
                    uint8_t *dst = reinterpret_cast<uint8_t *>(p.planes + word0 + (w0 >> 5)) + ((w0 & 31) >> 3);
                    if (p.tpw_log2 == 1) {
                        bw = squeeze2(bw); qw = squeeze2(qw);
                        *reinterpret_cast<uint16_t *>(dst) = (uint16_t)bw;
                        *reinterpret_cast<uint16_t *>(dst + 4) = (uint16_t)qw;
                    } else {
                        bw = squeeze4(bw); qw = squeeze4(qw);
                        dst[0] = (uint8_t)bw;
                        dst[4] = (uint8_t)qw;
                    }
                }
            } else {
                uint8_t *rb = resbuf + ((n * p.nsub + u) & 1) * kConsumerThreads;
                if (part == 0) rb[w] = (uint8_t)((bit ? 1 : 0) | (quiet ? 2 : 0));
                asm volatile("bar.sync 1, %0;" ::"n"(kConsumerThreads) : "memory");
                if (warp * 32 < wsub) {
                    const uint8_t r = rb[warp * 32 + lane];
                    const uint32_t bw = __ballot_sync(0xFFFFFFFFu, r & 1);
                    const uint32_t qw = __ballot_sync(0xFFFFFFFFu, r & 2);
                    if (lane == 0 && warp * 32 < nleft) p.planes[word0 + warp] = make_uint2(bw, qw);
                }
            }
        }
        }   // sub-tiles
        if (++s == S) { s = 0; ph ^= 1u; }
    }
    if (p.fused_frame) signal_finish(p, AS, sig, lane);
}

// ------------------------------------------------------------------------ k_demod_shift ----
// Short windows that are a multiple of 4 but not of 8 samples (bf = 12, 20: 4000 / 2400 baud).  One
// thread decodes kWpt consecutive windows (kBf * kWpt samples, a multiple of 8).  A window boundary
// then falls in the middle of a 16-byte vector; here the tile's alignment e (0..7, uniform over the tile) selects one of eight
// fully unrolled bodies in which the thread's words are picked at compile-time positions (even e:
// plain register renaming; odd e: one PRMT per word to splice the two half-words).  Every group of
// 4 samples lies inside one window (kBf % 4 == 0) and its +/-1 template weights are immediates.
__host__ __device__ constexpr uint32_t tone_weights4(int bf, int pos, bool space)
{
    // signed-byte weights of window samples pos .. pos+3: mark + - + - per quarter, space + + - -
    uint32_t w = 0;
    for (int s = 0; s < 4; s++) {
        const int qd = (pos + s) / (bf / 4);
        const bool neg = space ? (qd & 2) != 0 : (qd & 1) != 0;
        w |= (neg ? 0xFFu : 0x01u) << (8 * s);
    }
    return w;
}

template <int kBf, int kWpt, int kE, bool kPad>
__device__ __forceinline__ void shift_decode(const uint4 *dp, uint32_t k512, int thr_bf, int nvalid, uint32_t &bits,
                                             uint32_t &quiet)
{
    constexpr int kV = kBf * kWpt / 8;
    uint32_t W[4 * (kV + 1)];
#pragma unroll
    for (int i = 0; i <= kV; i++) {
        if (i < kV || kE > 0) {                      // an aligned tile never touches the extra vector
            const uint4 v = dp[(kPad && i == kV) ? kV + 1 : i];   // padded layout: the next segment starts one vector on
            W[4 * i] = v.x; W[4 * i + 1] = v.y; W[4 * i + 2] = v.z; W[4 * i + 3] = v.w;
        }
    }
#pragma unroll
    for (int w = 0; w < kWpt; w++) {
        int accM = 0, accS = 0, accA = 0;
        int UmF = 0, UsF = 0, NmF = 0, NsF = 0;      // windows of more than 120 samples: the packed sums are unpacked half way
#pragma unroll
        for (int b = 0; b < kBf / 4; b++) {
            if (kBf > 120 && b == kBf / 8) {
                unpack_acc(accM, UmF, NmF); unpack_acc(accS, UsF, NsF);
                accM = 0; accS = 0;
            }
            const int pos = kE + w * kBf + 4 * b;    // first sample of the group in the loaded words
            uint32_t a0, a1;
            if ((kE & 1) == 0) {
                a0 = W[pos / 2]; a1 = W[pos / 2 + 1];
            } else {
                a0 = prmt(W[(pos - 1) / 2], W[(pos + 1) / 2], 0x5432u);
                a1 = prmt(W[(pos + 1) / 2], W[(pos + 3) / 2], 0x5432u);
            }
            accum4_full(a0, a1, tone_weights4(kBf, 4 * b, false), tone_weights4(kBf, 4 * b, true), k512, accM, accS, accA);
        }
        // acc = 256 * T.n + T.c with |T.c| <= 127 (per half for long windows): decide as in k_demod
        const int Um = UmF + ((int)((unsigned)accM << 24) >> 24), Us = UsF + ((int)((unsigned)accS << 24) >> 24);
        const int du = Um - Us;
        bool b1 = du > 0;
        if (du == 0) {
            const int Nm = NmF + ((accM - ((int)((unsigned)accM << 24) >> 24)) >> 8);
            const int Ns = NsF + ((accS - ((int)((unsigned)accS << 24) >> 24)) >> 8);
            if (Ns > Nm) b1 = tie_bit(Um, Nm, Ns, kBf);
        }
        const bool valid = w < nvalid;
        bits |= (uint32_t)(valid && b1) << w;
        quiet |= (uint32_t)(valid && (accA < thr_bf)) << w;
    }
}

template <int kBf, int kWpt, bool kPad = false>
__global__ void __launch_bounds__(kFusedThreads4, 2) k_demod_shift(const DemodParams p)
{
    static_assert(kBf % 4 == 0 && (kBf * kWpt) % 8 == 0 && 32 % kWpt == 0, "segment must be whole vectors");
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int S = p.stages;
    uint8_t *stage_base = smem;
    TileMeta *meta = reinterpret_cast<TileMeta *>(smem + (size_t)S * p.stage_bytes);
    uint64_t *full = reinterpret_cast<uint64_t *>(meta + kMaxStages);
    uint64_t *empty = full + kMaxStages;
    constexpr int kSeg = kBf * kWpt, kLanesPerWord = 32 / kWpt;
    constexpr int kStride = kSeg / 8 + (kPad ? 1 : 0);       // vectors between the segments of consecutive threads

    if (tid == 0) {
        for (int s = 0; s < S; s++) {
            mbar_init(&full[s], kPad ? 32 * p.pad_warps + 1 : 1);
            mbar_init(&empty[s], kConsumerThreads / 32);
        }
        mbar_fence_init();
    }
    AuxSmem &AS = *reinterpret_cast<AuxSmem *>(smem + p.aux_off);
    aux_smem_init(p, AS);
    __syncthreads();

    const int ntile = (p.total_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles b, b + G, ...
    if (ntile <= 0) return;
    if constexpr (kPad) {
        // the producer warp and the (otherwise idle) auxiliary warps share the copies of every tile
        if (warp >= kConsumerThreads / 32) {
            const int pw = warp - kConsumerThreads / 32;
            if (pw < p.pad_warps) demod_produce_pad<kSeg / 8>(p, ntile, stage_base, meta, full, empty, pw, p.pad_warps);
            return;
        }
    }
    if (warp == kConsumerThreads / 32) {
        demod_produce(p, ntile, stage_base, meta, full, empty);
        return;
    }
    if (warp > kConsumerThreads / 32) {
        demod_aux<4>(p, smem);
        return;
    }
    TileSignal sig;

    const uint32_t k512 = 0x02000200u | ((uint32_t)p.stages >> 16);
    int s = 0;
    uint32_t ph = 0;
    for (int n = 0; n < ntile; ++n) {
        mbar_wait(&full[s], ph);
        const TileMeta m = meta[s];
        if (p.fused_frame) signal_note(p, AS, sig, m.gpos, m.want, lane);
#pragma unroll 1
        for (int u = 0; u < p.nsub; u++) {           // sub-tiles of kConsumerThreads * kWpt windows (see k_demod)
        const int wbase = u * kConsumerThreads * kWpt;
        uint32_t bits = 0, quiet = 0;
        if (m.nwin > wbase) {
            const uint4 *dp = reinterpret_cast<const uint4 *>(stage_base + (size_t)s * p.stage_bytes) + (m.e0 >> 3) +
                              (u * kConsumerThreads + tid) * kStride;
            const int nvalid = m.nwin - wbase - tid * kWpt;
            switch (m.e0 & 7) {                      // uniform over the CTA
            case 0: shift_decode<kBf, kWpt, 0, kPad>(dp, k512, m.thr_bf, nvalid, bits, quiet); break;
            case 1: shift_decode<kBf, kWpt, 1, kPad>(dp, k512, m.thr_bf, nvalid, bits, quiet); break;
            case 2: shift_decode<kBf, kWpt, 2, kPad>(dp, k512, m.thr_bf, nvalid, bits, quiet); break;
            case 3: shift_decode<kBf, kWpt, 3, kPad>(dp, k512, m.thr_bf, nvalid, bits, quiet); break;
            case 4: shift_decode<kBf, kWpt, 4, kPad>(dp, k512, m.thr_bf, nvalid, bits, quiet); break;
            case 5: shift_decode<kBf, kWpt, 5, kPad>(dp, k512, m.thr_bf, nvalid, bits, quiet); break;
            case 6: shift_decode<kBf, kWpt, 6, kPad>(dp, k512, m.thr_bf, nvalid, bits, quiet); break;
            default: shift_decode<kBf, kWpt, 7, kPad>(dp, k512, m.thr_bf, nvalid, bits, quiet); break;
            }
        }
        if (u == p.nsub - 1) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
        }
        if (m.nwin > wbase) {
            // kLanesPerWord threads hold the kWpt-bit pieces of one plane word
            uint32_t bw, qw;
            if (kWpt == 1) {                         // one window per lane: the plane words are warp ballots
                bw = __ballot_sync(0xFFFFFFFFu, bits != 0u);
                qw = __ballot_sync(0xFFFFFFFFu, quiet != 0u);
            } else {
                bw = bits << (kWpt * (lane & (kLanesPerWord - 1)));
                qw = quiet << (kWpt * (lane & (kLanesPerWord - 1)));
#pragma unroll
                for (int o = 1; o < kLanesPerWord; o <<= 1) {
                    bw |= __shfl_xor_sync(0xFFFFFFFFu, bw, o);
                    qw |= __shfl_xor_sync(0xFFFFFFFFu, qw, o);
                }
            }
            const int word = (tid * kWpt) >> 5;
            if ((lane & (kLanesPerWord - 1)) == 0 && word * 32 < m.nwin - wbase)
                p.planes[m.word_base + (wbase >> 5) + word] = make_uint2(bw, qw);
        }
        }   // sub-tiles
        if (++s == S) { s = 0; ph ^= 1u; }
    }
    if (p.fused_frame) signal_finish(p, AS, sig, lane);
}

// ------------------------------------------------------------------------- k_demod_lane ----
// Short windows of whole vectors (bf = 8, 16, 24: 6000 / 3000 / 2000 baud), lane-major: a consumer warp
// owns kJ * 32 consecutive windows of the tile and lane t decodes windows t, t + 32, ... of them, so the
// 128-bit loads of a warp are consecutive vectors (no bank conflicts, no rotation) and the 32 decisions of
// one step ARE a plane word (warp ballot).  The tile's alignment e (0..7, uniform over the tile because
// bf % 8 == 0) selects one of eight fully unrolled bodies: the window's words are picked at compile-time
// positions (even e: register renaming, odd e: one PRMT per word), the template weights are immediates,
// and the words of the first and last quarter of the bit — where mark and space agree, D = (mark -
// space) / 2 = 0 — are paired among themselves and only summed for the end detector (3 instead of 11
// instructions per 4 samples).
__host__ __device__ constexpr uint32_t d_weights4(int bf, int pos)
{
    // signed bytes of D = (mark - space) / 2 for window samples pos .. pos+3: 0, -1, +1, 0 per quarter
    uint32_t w = 0;
    for (int s = 0; s < 4; s++) {
        const int qd = (pos + s) / (bf / 4);
        w |= (qd == 1 ? 0xFFu : (qd == 2 ? 0x01u : 0x00u)) << (8 * s);
    }
    return w;
}

// the words of one window (samples 2i, 2i + 1 in X[i]) out of the vectors at v, for tile alignment kE
template <int kM, int kE>
__device__ __forceinline__ void lane_window_words(const uint4 *v, uint32_t (&X)[4 * kM])
{
    uint32_t W[4 * (kM + 1)];
#pragma unroll
    for (int i = 0; i <= kM; i++) {
        if (i < kM || kE > 0) {                      // an aligned tile never touches the extra vector
            const uint4 q = v[i];
            W[4 * i] = q.x; W[4 * i + 1] = q.y; W[4 * i + 2] = q.z; W[4 * i + 3] = q.w;
        }
    }
#pragma unroll
    for (int i = 0; i < 4 * kM; i++) {
        if ((kE & 1) == 0) X[i] = W[i + kE / 2];
        else X[i] = prmt(W[i + (kE - 1) / 2], W[i + (kE + 1) / 2], 0x5432u);
    }
}

template <int kM, int kJ, int kE>
__device__ __forceinline__ void lane_decode(const uint4 *dp, uint32_t k512, int thr_bf, uint32_t (&bw)[kJ], uint32_t (&qw)[kJ])
{
    constexpr int kBf = 8 * kM;
    const int lane = threadIdx.x & 31;
    uint32_t tb[kJ];
#pragma unroll
    for (int j = 0; j < kJ; j++) {
        uint32_t X[4 * kM];
        lane_window_words<kM, kE>(dp + j * 32 * kM, X);
        int accD = 0, accA = 0;
        // D = 0 outside samples [q, 3q) = words [q/2, 3q/2): those q words are classified in adjacent pairs,
        // the other q words (the first and last q/2) are paired among themselves for the amplitude only
        constexpr int kQ = kBf / 4, kH = kQ / 2;
#pragma unroll
        for (int k = 0; k < kH; k++)
            accum4_d(X[kH + 2 * k], X[kH + 2 * k + 1], d_weights4(kBf, kQ + 4 * k), k512, accD, accA);
#pragma unroll
        for (int k = 0; k < kH; k++) {
            // k-th pair of the list 0 .. q/2-1, 3q/2 .. 2q-1
            constexpr int kFirstHi = 3 * kH;
            const int a = 2 * k, b = 2 * k + 1;
            accum4_a(X[a < kH ? a : kFirstHi + (a - kH)], X[b < kH ? b : kFirstHi + (b - kH)], accA);
        }
        // accD = 256 * D.n + D.c, |D.c| <= bf / 2: D.c = (Um - Us) / 2 decides; when it is zero the window
        // is a 0 unless Ns > Nm (D.n < 0), and only then are the two floors compared (below)
        const int dl = (int)((unsigned)accD << 24);
        bw[j] = __ballot_sync(0xFFFFFFFFu, dl > 0);
        qw[j] = __ballot_sync(0xFFFFFFFFu, accA < thr_bf);
        tb[j] = __ballot_sync(0xFFFFFFFFu, dl == 0 && accD < 0);
    }
    // tied correlations (noise-only windows): the full mark / space sums decide, as in k_demod's plain mode
    uint32_t any = 0;
#pragma unroll
    for (int j = 0; j < kJ; j++) any |= tb[j];
    if (any) {
#pragma unroll 1
        for (int j = 0; j < kJ; j++) {
            uint32_t t = 0;
#pragma unroll
            for (int jj = 0; jj < kJ; jj++) t = (jj == j) ? tb[jj] : t;
            if (t == 0) continue;
            bool b1 = false;
            if ((t >> lane) & 1u) {
                uint32_t X[4 * kM];
                lane_window_words<kM, kE>(dp + j * 32 * kM, X);
                int accM = 0, accS = 0, accA = 0;
#pragma unroll
                for (int g = 0; g < 2 * kM; g++)
                    accum4_full(X[2 * g], X[2 * g + 1], tone_weights4(kBf, 4 * g, false), tone_weights4(kBf, 4 * g, true), k512,
                                accM, accS, accA);
                const int Um = (int)((unsigned)accM << 24) >> 24, Us = (int)((unsigned)accS << 24) >> 24;
                const int Nm = (accM - Um) >> 8, Ns = (accS - Us) >> 8;
                if (Um == Us && Ns > Nm) {
                    b1 = tie_bit(Um, Nm, Ns, kBf);
                } else {
                    b1 = Um > Us;
                }
            }
            const uint32_t fix = __ballot_sync(0xFFFFFFFFu, b1);
#pragma unroll
            for (int jj = 0; jj < kJ; jj++) bw[jj] |= (jj == j) ? fix : 0u;
        }
    }
}

template <int kM, int kJ, int kWarps>
__global__ void __launch_bounds__(kWarps * 32 + 32 + 128, 2) k_demod_lane(const DemodParams p)
{
    static_assert(kJ * 32 * kWarps * 8 * kM * 2 <= 64 * 1024, "tile");
    static_assert(kWarps * 32 == kConsumerThreads, "the auxiliary warps follow the producer warp");
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int S = p.stages;
    uint8_t *stage_base = smem;
    TileMeta *meta = reinterpret_cast<TileMeta *>(smem + (size_t)S * p.stage_bytes);
    uint64_t *full = reinterpret_cast<uint64_t *>(meta + kMaxStages);
    uint64_t *empty = full + kMaxStages;

    if (tid == 0) {
        for (int s = 0; s < S; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kWarps);
        }
        mbar_fence_init();
    }
    AuxSmem &AS = *reinterpret_cast<AuxSmem *>(smem + p.aux_off);
    aux_smem_init(p, AS);
    __syncthreads();

    const int ntile = (p.total_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles b, b + G, ...
    if (ntile <= 0) return;
    if (warp == kWarps) {
        demod_produce(p, ntile, stage_base, meta, full, empty);
        return;
    }
    if (warp > kWarps) {
        demod_aux<4>(p, smem);
        return;
    }
    TileSignal sig;

    const uint32_t k512 = 0x02000200u | ((uint32_t)p.stages >> 16);
    const int win0 = warp * kJ * 32;                  // first window of this warp in the tile
    int s = 0;
    uint32_t ph = 0;
    for (int n = 0; n < ntile; ++n) {
        mbar_wait(&full[s], ph);
        const TileMeta m = meta[s];
        if (p.fused_frame) signal_note(p, AS, sig, m.gpos, m.want, lane);
        uint32_t bw[kJ], qw[kJ];
#pragma unroll
        for (int j = 0; j < kJ; j++) { bw[j] = 0u; qw[j] = 0u; }
        const bool work = m.nwin > win0;              // warp-uniform: the warp has at least one valid window
        if (work) {
            const uint4 *dp = reinterpret_cast<const uint4 *>(stage_base + (size_t)s * p.stage_bytes) + (m.e0 >> 3) +
                              (win0 + lane) * kM;
            switch (m.e0 & 7) {                       // uniform over the CTA
            case 0: lane_decode<kM, kJ, 0>(dp, k512, m.thr_bf, bw, qw); break;
            case 1: lane_decode<kM, kJ, 1>(dp, k512, m.thr_bf, bw, qw); break;
            case 2: lane_decode<kM, kJ, 2>(dp, k512, m.thr_bf, bw, qw); break;
            case 3: lane_decode<kM, kJ, 3>(dp, k512, m.thr_bf, bw, qw); break;
            case 4: lane_decode<kM, kJ, 4>(dp, k512, m.thr_bf, bw, qw); break;
            case 5: lane_decode<kM, kJ, 5>(dp, k512, m.thr_bf, bw, qw); break;
            case 6: lane_decode<kM, kJ, 6>(dp, k512, m.thr_bf, bw, qw); break;
            default: lane_decode<kM, kJ, 7>(dp, k512, m.thr_bf, bw, qw); break;
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
        if (work && lane < kJ) {
            // lane j stores plane word j of the warp, windows past the capture's last one masked off
            uint32_t b = 0u, q = 0u;
#pragma unroll
            for (int j = 0; j < kJ; j++) { b = (lane == j) ? bw[j] : b; q = (lane == j) ? qw[j] : q; }
            const int nv = m.nwin - (win0 + 32 * lane);
            if (nv > 0) {
                const uint32_t vm = nv >= 32 ? 0xFFFFFFFFu : (1u << nv) - 1u;
                p.planes[m.word_base + (win0 >> 5) + lane] = make_uint2(b & vm, q & vm);
            }
        }
        if (++s == S) { s = 0; ph ^= 1u; }
    }
    if (p.fused_frame) signal_finish(p, AS, sig, lane);
}

// ------------------------------------------------------------------------------ k_frame ----
template <int kThreads, typename T>
__device__ __forceinline__ T block_min(T v, T *scratch)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    __syncthreads();                       // scratch reuse
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    T r = scratch[0];
#pragma unroll
    for (int w = 1; w < kThreads / 32; w++) r = min(r, scratch[w]);
    return r;
}

__device__ __forceinline__ uint32_t hamming74_nibble(uint32_t cw)
{
    // ECC.__decodeNibble :145-151 — cw bit i = c_i (c0 first received)
    const uint32_t s0 = __popc(cw & 0x55u) & 1u;   // c0^c2^c4^c6
    const uint32_t s1 = __popc(cw & 0x66u) & 1u;   // c1^c2^c5^c6
    const uint32_t s2 = __popc(cw & 0x78u) & 1u;   // c3^c4^c5^c6
    const uint32_t e = 4u * s2 + 2u * s1 + s0;
    if (e) cw ^= 1u << (e - 1u);
    return (((cw >> 2) & 1u) << 3) | (((cw >> 4) & 1u) << 2) | (((cw >> 5) & 1u) << 1) | ((cw >> 6) & 1u);
}

// two 7-bit codewords (14 bits, first received in bit 0) -> one byte, first nibble high (:393-399);
// lut[cw] = corrected nibble of codeword cw (128 entries, built per CTA)
__device__ __forceinline__ uint32_t decode_byte(uint32_t v14, const uint8_t *lut)
{

    return ((uint32_t)lut[v14 & 0x7Fu] << 4) | (uint32_t)lut[(v14 >> 7) & 0x7Fu];
}

// __scanTraining's terminator (:362-366) over plane word `cur` (decision bits of windows 32j .. 32j + 31) and the word
// before it: bit t is set when b[k-3] & ~b[k-2] & ~b[k-1] & ~b[k] for k = 32j + t
__device__ __forceinline__ uint32_t term_mask(uint32_t prev, uint32_t cur)
{
    return __funnelshift_l(prev, cur, 3) & ~__funnelshift_l(prev, cur, 2) & ~__funnelshift_l(prev, cur, 1) & ~cur;
}

// kThreads x kWords plane words are searched per block step: <128,4> for ordinary captures,
// <512,8> when the captures average more than 65536 windows (e.g. 64 KB payloads at 300 baud).
// idx_t = int unless a capture has 2^30 or more windows.
template <int kThreads, int kWords, typename idx_t>
__global__ void __launch_bounds__(kThreads) k_frame(const CapDesc *__restrict__ caps,
                                                    const int32_t *__restrict__ clock,
                                                    const uint2 *__restrict__ planes,
                                                    uint8_t *__restrict__ out,
                                                    AfskRxResult *__restrict__ res)
{
    const int c = blockIdx.x, tid = threadIdx.x;
    const CapDesc d = caps[c];
    if (d.status0 != 0) return;
    __shared__ idx_t scratch[kThreads / 32];
    __shared__ uint8_t lut[128];
    if (tid < 128) lut[tid] = (uint8_t)hamming74_nibble((uint32_t)tid);   // visible after the first block_min
    const int clk = clock[c];
    const idx_t K = (idx_t)num_windows(d.n, d.bf, clk);
    const idx_t nwords = (K + 31) >> 5;
    const uint2 *PL = planes + d.plane_base;
    const idx_t NONE = sizeof(idx_t) == 4 ? (idx_t)0x7FFFFFFF : (idx_t)0x7FFFFFFFFFFFFFFFLL;

    // phase 1 (:362-366): first k with bits[k-3..k] == 1,0,0,0 ; the shift register starts at 0
    idx_t kterm = NONE;
    for (idx_t base = 0; base < nwords; base += kThreads * kWords) {
        idx_t cand = NONE;
#pragma unroll
        for (int r = kWords - 1; r >= 0; r--) {
            const idx_t j = base + tid + r * kThreads;
            if (j < nwords) {
                const uint32_t cur = PL[j].x, prev = j ? PL[j - 1].x : 0u;
                uint32_t M = term_mask(prev, cur);
                const idx_t rem = K - 32 * j;
                if (rem < 32) M &= (1u << rem) - 1u;
                if (M) cand = 32 * j + (__ffs(M) - 1);
            }
        }
        kterm = block_min<kThreads, idx_t>(cand, scratch);
        if (kterm != NONE) break;
    }
    __syncthreads();                                 // lut (nwords may be 0: no block_min ran)
    const idx_t k0 = (kterm == NONE) ? K : kterm + 1;
    // phase 2 (:372-378): first quiet window at or after k0
    idx_t k1 = NONE;
    for (idx_t base = k0 >> 5; base < nwords; base += kThreads * kWords) {
        idx_t cand = NONE;
#pragma unroll
        for (int r = kWords - 1; r >= 0; r--) {
            const idx_t j = base + tid + r * kThreads;
            if (j < nwords) {
                uint32_t M = PL[j].y;
                if (j == (k0 >> 5)) M &= ~((1u << (k0 & 31)) - 1u);
                const idx_t rem = K - 32 * j;
                if (rem < 32) M &= (1u << rem) - 1u;
                if (M) cand = 32 * j + (__ffs(M) - 1);
            }
        }
        k1 = block_min<kThreads, idx_t>(cand, scratch);
        if (k1 != NONE) break;
    }
    if (k1 == NONE) k1 = K;
    const idx_t nbits = k1 - k0;
    const idx_t nbytes = (nbits / 7) / 2;            // ECC.decode :156, __bitsToBytes :396
    uint8_t *o = out + d.out_off;                    // 16-byte aligned
    // four bytes (56 coded bits) per thread step: three plane words, one 32-bit store
    const idx_t nquad = nbytes >> 2;
    for (idx_t i = tid; i < nquad; i += kThreads) {
        const idx_t pos = k0 + 56 * i;
        const idx_t wi = pos >> 5;
        const uint32_t sh = (uint32_t)(pos & 31);
        const uint32_t w0 = PL[wi].x, w1 = PL[wi + 1].x, w2 = PL[wi + 2].x;
        uint32_t word = 0;
#pragma unroll
        for (int jb = 0; jb < 4; jb++) {
            const uint32_t sft = sh + 14u * jb;                 // 0 .. 73
            const uint32_t a = sft < 32 ? w0 : (sft < 64 ? w1 : w2);
            const uint32_t bb = sft < 32 ? w1 : (sft < 64 ? w2 : 0u);
            word |= decode_byte(__funnelshift_r(a, bb, sft & 31u) & 0x3FFFu, lut) << (8 * jb);
        }
        reinterpret_cast<uint32_t *>(o)[i] = word;
    }
    for (idx_t i = 4 * nquad + tid; i < nbytes; i += kThreads) {
        const idx_t pos = k0 + 14 * i;
        const uint32_t lo = PL[pos >> 5].x, hi = PL[(pos >> 5) + 1].x;
        o[i] = (uint8_t)decode_byte(__funnelshift_r(lo, hi, (uint32_t)(pos & 31)) & 0x3FFFu, lut);
    }
    if (tid == 0) {
        AfskRxResult r;
        r.status = nbits > 0 ? AFSK_ST_OK : AFSK_ST_NO_DATA;
        r.clock = clk;
        r.train_end = (long long)clk + (long long)k0 * d.bf;   // "Training sequence terminated on frame" :368
        r.nbits = nbits;
        r.nbytes = nbits > 0 ? nbytes : 0;
        res[c] = r;
    }
}

// One WARP per capture (four captures per CTA) for batches of ordinary captures: the two find-first
// searches reduce with one REDUX per step instead of a CTA-wide barrier pair, no shared scratch, and
// four times as many captures are in flight per SM.  Same arithmetic as k_frame above; used when no
// capture of the batch has more than kFrameWarpMaxWindows windows.
constexpr int kFrameWarpCaps = 4;                      // warps (captures) per CTA
constexpr int64_t kFrameWarpMaxWindows = 262144;       // 8192 plane words: 64 search steps of one warp

// kCg: the plane words were written by other CTAs of the same launch (fused mode): read them from L2.
template <bool kCg>
__device__ __forceinline__ uint32_t plane_word(const uint32_t *p)
{
    return kCg ? ld_cg_u32(p) : *p;
}

// framing of one capture by one warp: the body of k_frame_warp and of the fused kernel's frame jobs
template <bool kCg>
__device__ __forceinline__ void frame_capture_warp(int c, const CapDesc &d, int clk, const uint2 *__restrict__ planes,
                                                   uint8_t *__restrict__ out, AfskRxResult *__restrict__ res,
                                                   const uint8_t *lut, int lane)
{
    const int K = (int)num_windows(d.n, d.bf, clk);
    const int nwords = (K + 31) >> 5;
    const uint32_t *PW = reinterpret_cast<const uint32_t *>(planes + d.plane_base);   // word j: bits PW[2j], quiet PW[2j + 1]
    constexpr unsigned NONE = 0x7FFFFFFFu;
    constexpr int kWords = 8;                           // plane words per lane per step (loads in flight)
    AFSK_TRACE_DECL
    AFSK_TRACE_MARK

    // Every step issues all of its loads before it looks at any of them: a frame job of the fused kernel runs
    // on one warp beside a saturated memory system, where a dependent L2 round trip costs microseconds.
    // phase 1 (:362-366): first k with bits[k-3..k] == 1,0,0,0 ; the shift register starts at 0
    unsigned kterm = NONE;
    for (int base = 0; base < nwords; base += 32 * kWords) {
        uint32_t cur[kWords], prv[kWords];
#pragma unroll
        for (int r = 0; r < kWords; r++) {
            const int j = base + lane + 32 * r;
            cur[r] = j < nwords ? plane_word<kCg>(PW + 2 * j) : 0u;
            prv[r] = (j < nwords && j > 0) ? plane_word<kCg>(PW + 2 * j - 2) : 0u;
        }
        unsigned cand = NONE;
#pragma unroll
        for (int r = kWords - 1; r >= 0; r--) {
            const int j = base + lane + 32 * r;
            if (j < nwords) {
                uint32_t M = term_mask(prv[r], cur[r]);
                const int rem = K - 32 * j;
                if (rem < 32) M &= (1u << rem) - 1u;
                if (M) cand = (unsigned)(32 * j + (__ffs(M) - 1));
            }
        }
        kterm = __reduce_min_sync(0xFFFFFFFFu, cand);
        if (kterm != NONE) break;
    }
    const int k0 = (kterm == NONE) ? K : (int)kterm + 1;
    AFSK_TRACE_MARK
    // phase 2 (:372-378): first quiet window at or after k0
    unsigned kq = NONE;
    for (int base = k0 >> 5; base < nwords; base += 32 * kWords) {
        uint32_t qw[kWords];
#pragma unroll
        for (int r = 0; r < kWords; r++) {
            const int j = base + lane + 32 * r;
            qw[r] = j < nwords ? plane_word<kCg>(PW + 2 * j + 1) : 0u;
        }
        unsigned cand = NONE;
#pragma unroll
        for (int r = kWords - 1; r >= 0; r--) {
            const int j = base + lane + 32 * r;
            if (j < nwords) {
                uint32_t M = qw[r];
                if (j == (k0 >> 5)) M &= ~((1u << (k0 & 31)) - 1u);
                const int rem = K - 32 * j;
                if (rem < 32) M &= (1u << rem) - 1u;
                if (M) cand = (unsigned)(32 * j + (__ffs(M) - 1));
            }
        }
        kq = __reduce_min_sync(0xFFFFFFFFu, cand);
        if (kq != NONE) break;
    }
    const int k1 = (kq == NONE) ? K : (int)kq;
    AFSK_TRACE_MARK
    const int nbits = k1 - k0;
    const int nbytes = (nbits / 7) / 2;              // ECC.decode :156, __bitsToBytes :396
    uint8_t *o = out + d.out_off;                    // 16-byte aligned
    // four bytes (56 coded bits) per lane step: three plane words, one 32-bit store; four steps' loads at a time
    const int nquad = nbytes >> 2;
    constexpr int kQ = 4;
    for (int i0 = lane; i0 < nquad; i0 += 32 * kQ) {
        uint32_t w[kQ][3];
#pragma unroll
        for (int u = 0; u < kQ; u++) {
            const int i = i0 + 32 * u;
            const int wi = (k0 + 56 * i) >> 5;
#pragma unroll
            for (int t = 0; t < 3; t++) w[u][t] = i < nquad ? plane_word<kCg>(PW + 2 * (wi + t)) : 0u;
        }
#pragma unroll
        for (int u = 0; u < kQ; u++) {
            const int i = i0 + 32 * u;
            if (i < nquad) {
                // the quad's 56 coded bits as a stream (v: bits 0..31, v1: bits 32..63), eight 7-bit codewords cut out of it
                const uint32_t sh = (uint32_t)((k0 + 56 * i) & 31);
                const uint32_t v = __funnelshift_r(w[u][0], w[u][1], sh), v1 = __funnelshift_r(w[u][1], w[u][2], sh);
                const uint32_t n0 = lut[v & 0x7Fu], n1 = lut[(v >> 7) & 0x7Fu], n2 = lut[(v >> 14) & 0x7Fu], n3 = lut[(v >> 21) & 0x7Fu];
                const uint32_t n4 = lut[__funnelshift_r(v, v1, 28) & 0x7Fu], n5 = lut[(v1 >> 3) & 0x7Fu];
                const uint32_t n6 = lut[(v1 >> 10) & 0x7Fu], n7 = lut[(v1 >> 17) & 0x7Fu];
                // first nibble of a byte high (:393-399), bytes little-endian in the stored word
                reinterpret_cast<uint32_t *>(o)[i] = (n0 << 4) | n1 | (n2 << 12) | (n3 << 8) | (n4 << 20) | (n5 << 16) | (n6 << 28) | (n7 << 24);
            }
        }
    }
    for (int i = 4 * nquad + lane; i < nbytes; i += 32) {
        const int pos = k0 + 14 * i;
        const uint32_t lo = plane_word<kCg>(PW + 2 * (pos >> 5)), hi = plane_word<kCg>(PW + 2 * (pos >> 5) + 2);
        o[i] = (uint8_t)decode_byte(__funnelshift_r(lo, hi, (uint32_t)(pos & 31)) & 0x3FFFu, lut);
    }
    AFSK_TRACE_MARK
    if ((c & 7) == 0) { AFSK_TRACE_EMIT((kCg ? 2ull : 3ull) + ((unsigned long long)blockIdx.x << 8)) }
    if (lane == 0) {
        AfskRxResult r;
        r.status = nbits > 0 ? AFSK_ST_OK : AFSK_ST_NO_DATA;
        r.clock = clk;
        r.train_end = (long long)clk + (long long)k0 * d.bf;   // "Training sequence terminated on frame" :368
        r.nbits = nbits;
        r.nbytes = nbits > 0 ? nbytes : 0;
        res[c] = r;
    }
}

__global__ void __launch_bounds__(32 * kFrameWarpCaps) k_frame_warp(const CapDesc *__restrict__ caps,
                                                                    const int32_t *__restrict__ clock,
                                                                    const uint2 *__restrict__ planes,
                                                                    uint8_t *__restrict__ out,
                                                                    AfskRxResult *__restrict__ res, int B)
{
    const int tid = threadIdx.x, lane = tid & 31;
    __shared__ uint8_t lut[128];
    static_assert(32 * kFrameWarpCaps == 128, "one LUT entry per thread");
    lut[tid] = (uint8_t)hamming74_nibble((uint32_t)tid);
    __syncthreads();
    const int c = blockIdx.x * kFrameWarpCaps + (tid >> 5);
    if (c >= B) return;
    const int clk = clock[c];                          // issued together with the descriptor load
    const CapDesc d = caps[c];
    if (d.status0 != 0) return;
    frame_capture_warp<false>(c, d, clk, planes, out, res, lut, lane);
}

// results of the captures that are decided on the host (exceptions, too short): the fused path has no k_clock
__global__ void __launch_bounds__(256) k_preset(const CapDesc *__restrict__ caps, int32_t *__restrict__ clock,
                                                AfskRxResult *__restrict__ res, int B)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= B) return;
    const int st = caps[c].status0;
    if (st == 0) return;
    clock[c] = -1;
    AfskRxResult r;
    r.status = st; r.clock = -1; r.train_end = -1; r.nbits = 0; r.nbytes = 0;
    res[c] = r;
}

// The auxiliary warps of one CTA of a fused demodulator launch (see "auxiliary warps" above).
// Framing is dealt out statically: auxiliary warp gw of the launch (gw = CTA * kAW + warp) frames captures
// gw, gw + W, gw + 2W, ... of the group (W = auxiliary warps of the whole launch), in that order, each as soon
// as its tile counter shows every tile reported.  (Measured alternatives: letting the CTA whose report
// completes a capture frame it hands hundreds of captures to the one CTA that reports last in every report
// interval; one launch-wide queue popped by compare-and-swap collapses under 1,184 pollers.)
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// frames capture position ci if all of its tiles have been reported; false otherwise (nothing waits here)
__device__ __forceinline__ bool aux_try_frame(const DemodParams &p, AuxSmem &S, int ci, int lane)
{
    uint32_t ready = 0;
    if (lane == 0) {
        const uint32_t want = (uint32_t)(p.gtile_first[ci + 1] - p.gtile_first[ci]);
        ready = ld_acquire_u32(p.tiles_done + ci) == want;        // acquire: every CTA's plane words of the capture
        if (ready) p.tiles_done[ci] = 0u;                          // nobody touches the counter again in this launch
    }
    if (!__shfl_sync(0xFFFFFFFFu, ready, 0)) return false;
    const int c = p.gcaps[ci];
    const CapDesc d = p.caps[c];
    const int clk = (int)(uint32_t)ld_relaxed_u64(p.cready + c);
#ifndef AFSK_DBG_NOFRAME
    frame_capture_warp<true>(c, d, clk, p.planes, p.out, p.res, S.lut, lane);
#endif
    return true;
}

template <int kAW>
__device__ __forceinline__ void demod_aux(const DemodParams &p, uint8_t *smem)
{
    constexpr int kAT = 32 * kAW;
    AuxSmem &S = *reinterpret_cast<AuxSmem *>(smem + p.aux_off);
    const int atid = (int)threadIdx.x - kDemodThreads, lane = atid & 31;
    uint32_t *ctrl = p.ctrl + 4 * (p.epoch & 1u);
    if (blockIdx.x == 0 && atid == 0) {               // the other slot serves the next launch of this group
        uint32_t *other = p.ctrl + 4 * ((p.epoch + 1u) & 1u);
        other[0] = 0u;
    }
    if (p.fused_frame)                                // Hamming(7,4) nibble table; visible after the first aux_bar below
        for (int i = atid; i < 128; i += kAT) S.lut[i] = (uint8_t)hamming74_nibble((uint32_t)i);
    // this warp's framing list: captures fnext, fnext + fstride, ... of the group
    const int fstride = (int)gridDim.x * kAW;
    int fnext = (int)blockIdx.x * kAW + (atid >> 5);
    // ---- clock jobs, in capture order, the auxiliary warps of the CTA together; between two clock jobs
    //      every warp frames the next capture of its list if that one is complete ----
    for (int it = 0;; it++) {
        if (atid == 0) S.job[it & 1] = (int)atomicAdd(&ctrl[0], 1u);
        aux_bar<kAW>();
        const int j = S.job[it & 1];
        if (j >= p.ng) break;
        const int c = p.gcaps[j];
        const long long off = p.caps[c].off;
        AFSK_TRACE_DECL
        AFSK_TRACE_MARK
        const uint32_t clk = aux_clock_index<kAW>(p.samples, off, p.bf, p.clk_magic, p.clk_shift, S, atid);
        AFSK_TRACE_MARK
        if (atid == 0) { AFSK_TRACE_EMIT(1ull) }
        if (atid == 0) {
            p.clock_out[c] = (int32_t)clk;
            st_relaxed_u64(p.cready + c, ((unsigned long long)p.epoch << 32) | clk);
        }
        if (p.fused_frame && fnext < p.ng && aux_try_frame(p, S, fnext, lane)) fnext += fstride;
    }
    if (!p.fused_frame) return;
    // ---- the rest of the list.  A capture completes when the consumer warps of every CTA holding one of its
    //      tiles have reported: this waits for other CTAs, all of which are resident (the grid is sized to
    //      the device's capacity for this kernel). ----
    uint32_t backoff = 100;
    unsigned long long t0 = 0;
    while (fnext < p.ng) {
        if (aux_try_frame(p, S, fnext, lane)) { fnext += fstride; backoff = 100; t0 = 0; continue; }
        __nanosleep(backoff);
        spin_guard(t0);
        backoff = backoff < 1600 ? backoff * 2 : backoff;
    }
    {
        AFSK_TRACE_DECL
        AFSK_TRACE_MARK
        AFSK_TRACE_MARK
        if (atid == 0) { AFSK_TRACE_EMIT(6ull + ((unsigned long long)blockIdx.x << 8)) }
    }
}

// Consumer side of fused framing.  Reporting a finished tile to its capture's counter needs a release at
// GPU scope (the plane words must be visible to whichever CTA frames the capture).  A fence per tile and
// warp costs more than the tile, and one atomic per tile and warp crowds the L2 atomic unit of the few
// counters the whole grid is working on.  So a consumer warp only NOTES its tiles (signal_note, one per
// lane) and reports 32 at a time: fence (its own plane stores), then every lane arrives on the tile's slot in
// shared memory; the lane whose arrival is the CTA's last for the tile (all consumer warps have fenced and
// arrived) fences again (the arrivals it observed -> its own report) and adds ONE to the capture's counter.
__device__ __forceinline__ void signal_flush(const DemodParams &p, AuxSmem &S, TileSignal &t, int lane)
{
    if (t.npend == 0) return;
    __syncwarp();                                     // the other lanes' plane stores
    asm volatile("fence.acq_rel.gpu;" ::: "memory");
    const bool mine = lane < t.npend;
    bool cta_last = false;
    uint32_t *slot = &S.tile_arr[(t.n0 + lane) % kAuxTileSlots];
    if (mine) cta_last = atomicAdd(slot, 1u) == (uint32_t)(kConsumerThreads / 32 - 1);
    if (__any_sync(0xFFFFFFFFu, cta_last)) {
        asm volatile("fence.acq_rel.gpu;" ::: "memory");
        if (cta_last) {
            *slot = 0u;                               // the slot's next user is kAuxTileSlots tiles away
            asm volatile("red.relaxed.gpu.global.add.u32 [%0], 1;" ::"l"(p.tiles_done + t.ci) : "memory");
        }
    }
    __syncwarp();
    t.npend = 0;
}

// after a consumer warp's last tile
__device__ __forceinline__ void signal_finish(const DemodParams &p, AuxSmem &S, TileSignal &t, int lane)
{
    signal_flush(p, S, t, lane);
}

// ------------------------------------------------------------------------------- k_gate ----
// Receiver.__listen (:299-319) arithmetic: per-2048-frame chunk amplitude, then open/close search.
__global__ void __launch_bounds__(256) k_gate_amp(const int16_t *__restrict__ x, const int64_t *__restrict__ chunk_first,
                                                  const int64_t *__restrict__ off, int S, long long total_chunks,
                                                  int32_t *__restrict__ amp)
{
    const int lane = threadIdx.x & 31;
    const long long gw = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (gw >= total_chunks) return;
    int a = 0, b = S;                       // stream of this chunk
    while (b - a > 1) {
        const int mid = (a + b) >> 1;
        if (chunk_first[mid] <= gw) a = mid; else b = mid;
    }
    // the chunk as 16-byte vectors from the aligned address at or below its first frame: 256 vectors,
    // or 257 with the frames outside the chunk masked off when it starts mid-vector
    const long long g0 = off[a] + (gw - chunk_first[a]) * AFSK_GATE_CHUNK;
    const int e = (int)(g0 & 7);
    const uint4 *src = reinterpret_cast<const uint4 *>(x + (g0 - e));
    const int nvec = AFSK_GATE_CHUNK / 8 + (e ? 1 : 0);
    int acc = 0;
    for (int v = lane; v < nvec; v += 32) {
        const uint4 qv = ld_nc_v4(src + v);
        // sign(x) per frame as a signed byte (+1 / -1), zero outside [g0, g0 + 2048): sum sign(x) * x = sum |x|
        uint32_t sa = prmt(qv.x, qv.y, 0xFDB9u) | 0x01010101u, sb = prmt(qv.z, qv.w, 0xFDB9u) | 0x01010101u;
        if (v == 0 && e) {
            const unsigned long long keep = ~0ull << (8 * e);
            sa &= (uint32_t)keep; sb &= (uint32_t)(keep >> 32);
        }
        if (v == AFSK_GATE_CHUNK / 8) {          // only reached when e > 0: frames 0 .. e-1 of the last vector
            const unsigned long long keep = ~(~0ull << (8 * e));
            sa &= (uint32_t)keep; sb &= (uint32_t)(keep >> 32);
        }
        acc = __dp2a_lo((int)qv.x, (int)sa, acc);
        acc = __dp2a_hi((int)qv.y, (int)sa, acc);
        acc = __dp2a_lo((int)qv.z, (int)sb, acc);
        acc = __dp2a_hi((int)qv.w, (int)sb, acc);
    }
    uint32_t sum = (uint32_t)acc;             // <= 2048 * 32768 = 2^26
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xFFFFFFFFu, sum, o);
    if (lane == 0) amp[gw] = (int32_t)(sum / AFSK_GATE_CHUNK);          // getAmplitude :94-98
}

__global__ void __launch_bounds__(kFrameThreads) k_gate_scan(const int32_t *__restrict__ amp,
                                                             const int64_t *__restrict__ chunk_first, int amp_start,
                                                             int amp_end, long long timeout_frames,
                                                             int64_t *__restrict__ range)
{
    const int s = blockIdx.x, tid = threadIdx.x;
    __shared__ long long scratch[kFrameThreads / 32];
    const long long NONE = 0x7FFFFFFFFFFFFFFFLL;
    const int32_t *A = amp + chunk_first[s];
    const long long nch = chunk_first[s + 1] - chunk_first[s];
    // chunk idx >= 1 is examined iff (idx-1)*2048 < timeout_frames  (:304,:310)
    long long lim = timeout_frames <= 0 ? 0 : (timeout_frames + AFSK_GATE_CHUNK - 1) / AFSK_GATE_CHUNK;  // idx <= lim
    long long last = min(nch - 1, lim);
    long long open = NONE;
    for (long long base = 1; base <= last; base += kFrameThreads) {
        const long long j = base + tid;
        long long cand = (j <= last && A[j] > amp_start) ? j : NONE;     // :306
        open = block_min<kFrameThreads, long long>(cand, scratch);
        if (open != NONE) break;
    }
    long long close = NONE;
    if (open != NONE) {
        for (long long base = open + 1; base < nch; base += kFrameThreads) {
            const long long j = base + tid;
            long long cand = (j < nch && A[j] < amp_end) ? j : NONE;     // :316
            close = block_min<kFrameThreads, long long>(cand, scratch);
            if (close != NONE) break;
        }
    }
    if (tid == 0) {
        if (open == NONE) {
            range[3 * s] = 0; range[3 * s + 1] = 0; range[3 * s + 2] = 0;
        } else {
            range[3 * s] = 1;
            range[3 * s + 1] = open * AFSK_GATE_CHUNK;
            range[3 * s + 2] = (close == NONE ? (nch > open + 1 ? nch : open + 1) : close + 1) * AFSK_GATE_CHUNK;
        }
    }
}

// Successive Receiver.receive() calls over one stream (the reference keeps its input stream open
// between calls, afskmodem.py:283): every call discards one chunk (:303), examines up to
// ceil(timeout / 2048) chunks for an opening (:304-310) and, once open, records through the first
// chunk quieter than amp_end (:313-318); the next call starts at the chunk after.  One warp per
// stream walks the chunk amplitudes 32 at a time.
//
// The walk is resumable: it starts from a saved GateState (afsk_rx_gate_multi: a fresh one) over the
// chunks that arrived since, emits only the calls that became final (timed out with all their chunks
// present, or closed by a quiet chunk) and saves where it stopped.  After every walk `pos` equals the
// number of chunks seen, so the next walk needs the amplitudes of the new chunks only.  finish applies
// the finite-stream conventions: a recording still open keeps everything up to the last full chunk;
// a call that has neither opened nor timed out does not return.
struct GateState {
    long long pos;      // next chunk to read
    long long mark;     // phase 1: first chunk the call listens at; phase 2: chunk that opened the recording
    long long call;     // calls finished so far
    int phase;          // 0: the call discards chunk `pos` first; 1: listening; 2: recording
    int pad;
};
static_assert(sizeof(GateState) == 32, "GateState layout");
__device__ __forceinline__ long long warp_find_first(const int32_t *A, long long lo, long long hi, int thr, bool greater)
{
    const int lane = threadIdx.x & 31;
    for (long long base = lo; base < hi; base += 32) {
        const long long j = base + lane;
        bool hit = false;
        if (j < hi) {
            const int a = A[j];
            hit = greater ? (a > thr) : (a < thr);
        }
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, hit);
        if (m) return base + (__ffs(m) - 1);
    }
    return -1;
}

// One receiver's gate settings (Receiver amp_start / amp_end thresholds, receive() timeout in frames).
struct GateParams {
    int amp_start, amp_end;
    long long timeout_frames;
};
static_assert(sizeof(GateParams) == 16, "GateParams layout");

// amp[chunk_first[s] ..] are the amplitudes of stream s's chunks from state[s].pos on (state == NULL: a
// fresh state).  Stream s gates with params[s] (params == NULL: `uni` for every stream) and finishes when
// fin[s] != 0 (fin == NULL: when `finish`); a finished stream's state is reset to a fresh one.  Call k of
// this walk goes to ranges[3 * (out_first ? out_first[s] : s * max_calls) + 3k].  Every call emitted before
// finish reads at least one new chunk, so new chunks + 1 slots always suffice.
__global__ void __launch_bounds__(32) k_gate_multi(const int32_t *__restrict__ amp, const int64_t *__restrict__ chunk_first,
                                                   GateParams uni, const GateParams *__restrict__ params, int max_calls,
                                                   GateState *__restrict__ state, int finish, const uint8_t *__restrict__ fin,
                                                   const int64_t *__restrict__ out_first, int64_t *__restrict__ ranges,
                                                   int32_t *__restrict__ counts)
{
    const int s = blockIdx.x, lane = threadIdx.x;
    const GateParams p = params ? params[s] : uni;
    const int amp_start = p.amp_start, amp_end = p.amp_end;
    if (fin) finish = fin[s];
    GateState g = {0, 0, 0, 0, 0};
    if (state) g = state[s];
    const int32_t *A = amp + chunk_first[s] - g.pos;             // A[j]: chunk j of the stream
    const long long nch = g.pos + chunk_first[s + 1] - chunk_first[s];
    const long long lim = p.timeout_frames <= 0 ? 0 : (p.timeout_frames + AFSK_GATE_CHUNK - 1) / AFSK_GATE_CHUNK;
    int64_t *out = ranges + (out_first ? (long long)out_first[s] : (long long)s * max_calls) * 3;
    int calls = 0;
    while (calls < max_calls) {
        if (g.phase == 0) {
            if (g.pos >= nch) break;
            g.pos++;                                              // chunk discarded :303
            g.phase = 1; g.mark = g.pos;
        }
        long long rec = 0, a = 0, b = 0;
        if (g.phase == 1) {
            const long long stop = g.mark + lim;
            const long long open = warp_find_first(A, g.pos, min(stop, nch), amp_start, true);     // :306
            if (open < 0) {
                if (stop > nch) { g.pos = nch; break; }           // not timed out yet
                g.pos = stop;                                     // "Timed out." :311-312, :405-407
            } else {
                g.phase = 2; g.mark = open; g.pos = open + 1;
            }
        }
        if (g.phase == 2) {
            const long long close = warp_find_first(A, g.pos, nch, amp_end, false);                 // :316
            if (close < 0) { g.pos = nch; break; }                // still recording
            rec = 1; a = g.mark * AFSK_GATE_CHUNK; b = (close + 1) * AFSK_GATE_CHUNK;
            g.pos = close + 1;
        }
        if (lane == 0) { out[3 * calls] = rec; out[3 * calls + 1] = a; out[3 * calls + 2] = b; }
        calls++;
        g.phase = 0;
    }
    if (finish && g.phase == 2 && calls < max_calls) {
        if (lane == 0) { out[3 * calls] = 1; out[3 * calls + 1] = g.mark * AFSK_GATE_CHUNK; out[3 * calls + 2] = nch * AFSK_GATE_CHUNK; }
        calls++;
        g.phase = 0;
    }
    g.call += calls;
    if (lane == 0) {
        counts[s] = calls;
        if (state) state[s] = finish ? GateState{0, 0, 0, 0, 0} : g;
    }
}

// Copies segments of samples between buffers at any frame alignment, one launch for all of them: every
// thread writes one aligned 16-byte vector of the destination from the (at most two) aligned source
// vectors that hold its frames, realigned with funnel shifts.  Only the partial head and tail vectors
// of a segment are written frame by frame (the frames around them belong to other data).
struct CopySeg { long long src, dst, len; };                     // samples
constexpr int kCopyThreads = 256, kCopyTileVecs = 4 * kCopyThreads;

// samples k .. k + 7 of the sixteen in two consecutive aligned vectors
__device__ __forceinline__ void realign8(const uint4 &lo, const uint4 &hi, int k, uint32_t (&o)[4])
{
    const uint32_t w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    const int j = k >> 1;
#pragma unroll
    for (int t = 0; t < 4; t++) {
        const uint32_t x0 = j == 0 ? w[t] : j == 1 ? w[t + 1] : j == 2 ? w[t + 2] : w[t + 3];
        const uint32_t x1 = j == 0 ? w[t + 1] : j == 1 ? w[t + 2] : j == 2 ? w[t + 3] : w[t + 4];
        o[t] = (k & 1) ? __funnelshift_r(x0, x1, 16) : x0;
    }
}

__global__ void __launch_bounds__(kCopyThreads) k_stream_copy(const int16_t *__restrict__ src, int16_t *__restrict__ dst,
                                                              const CopySeg *__restrict__ seg,
                                                              const int64_t *__restrict__ tile_first, int n)
{
    const long long tile = blockIdx.x;
    int a = 0, b = n;                                             // segment of this tile
    while (b - a > 1) {
        const int mid = (a + b) >> 1;
        if (tile_first[mid] <= tile) a = mid; else b = mid;
    }
    const CopySeg g = seg[a];
    const long long v0 = (g.dst >> 3) + (tile - tile_first[a]) * kCopyTileVecs, vend = (g.dst + g.len + 7) >> 3;
    const long long s_lo = g.src >> 3, s_hi = (g.src + g.len - 1) >> 3;
#pragma unroll
    for (int i = 0; i < kCopyTileVecs / kCopyThreads; i++) {
        const long long dv = v0 + i * kCopyThreads + threadIdx.x;
        if (dv >= vend) break;
        const long long q = dv * 8 - g.dst + g.src;               // source frame of the vector's first frame
        const long long sv = q >> 3;                              // (floor: q < 0 only at a head vector)
        const int k = (int)(q - sv * 8);
        uint4 lo = make_uint4(0, 0, 0, 0), hi = make_uint4(0, 0, 0, 0);
        if (sv >= s_lo && sv <= s_hi) lo = ld_nc_v4(src + sv * 8);
        if (k && sv + 1 >= s_lo && sv + 1 <= s_hi) hi = ld_nc_v4(src + (sv + 1) * 8);
        uint32_t o[4];
        realign8(lo, hi, k, o);
        const long long d0 = dv * 8;
        if (d0 >= g.dst && d0 + 8 <= g.dst + g.len) {
            *reinterpret_cast<uint4 *>(dst + d0) = make_uint4(o[0], o[1], o[2], o[3]);
        } else {
#pragma unroll
            for (int e = 0; e < 8; e++)
                if (d0 + e >= g.dst && d0 + e < g.dst + g.len) dst[d0 + e] = (int16_t)(o[e >> 1] >> (16 * (e & 1)));
        }
    }
}

// k_stream_frames<Tin> appends one interleaved piece to every channel's slot: frame f of channel s is element
// e0 + f * pitch + s of src
// (src 16-byte aligned, e0 < 16 / sizeof(Tin) the window's offset in its first vector, pitch >= S, n frames), converted
// to int16 by the rule of its format (sample_to_s16) as it is loaded; it goes to dst[seg[s].dst + f], an arbitrary
// alignment per channel.  A CTA owns kDiC consecutive channels x kDiF destination frames, in destination-vector
// coordinates: tile fb writes channel s's vectors (seg[s].dst >> 3) + fb * kDiF / 8 + j, j < kDiF / 8, which hold
// frames fb * kDiF - a + 8j .. + 7 with a = seg[s].dst & 7.  So the tile reads frame rows fb * kDiF - 7 .. fb * kDiF +
// kDiF - 1 (a halo of 7 frames in front), each row's kDiC channels as contiguous bytes with aligned 128-bit loads,
// realigned to the window with funnel shifts (16-bit) or word selects (32-bit): only the vectors holding window
// samples are read.  A 16-bit row is 128 bytes, eight lanes of 8 samples; a 32-bit row is 256 bytes, sixteen lanes of
// 4 samples, so that every load instruction still covers whole 128-byte lines and the tile, its shared layout and the
// store half stay those of the 16-bit case.  Each frame lands in shared memory at its channel's destination position,
// so every thread then writes aligned 16-byte vectors of one channel, sixteen lanes one 256-byte run; only a channel's
// head and tail vectors are written frame by frame.  64 x 128 keeps the tile at 17 KB (several CTAs per SM); the halo
// costs 7 / 128 extra reads.  Shared rows are channels in the order (s & 7) * 8 + (s >> 3), 136 samples apart (68 words
// = 4 banks): the eight lanes of a 16-bit row load write eight consecutive rows, in disjoint bank groups (a 32-bit row's
// sixteen lanes fall on eight bank groups, two lanes each).
constexpr int kDiC = 64, kDiF = 128, kDiHalo = 7, kDiThreads = 256, kDiStride = kDiF + 8;

__device__ __forceinline__ int di_row(int c) { return (c & 7) * 8 + (c >> 3); }

// k_stream_frames<int16_t> for contiguous frames of a 16-byte aligned piece (pitch S, e0 = 0), the layout of
// afsk_rx_streams_push_interleaved: its row arithmetic is cheaper, and it measured faster (DESIGN.md §5)
__global__ void __launch_bounds__(kDiThreads) k_stream_deinterleave(const int16_t *__restrict__ src, int16_t *__restrict__ dst,
                                                                     const CopySeg *__restrict__ seg, int S, long long n,
                                                                     int cblocks)
{
    __shared__ __align__(16) int16_t T[kDiC * kDiStride];
    __shared__ long long sdst[kDiC];
    const int c0 = (int)(blockIdx.x % cblocks) * kDiC, nc = min(kDiC, S - c0);
    const long long F0 = (long long)(blockIdx.x / cblocks) * kDiF;
    if (threadIdx.x < nc) sdst[threadIdx.x] = seg[c0 + threadIdx.x].dst;
    __syncthreads();
    const long long f_lo = max(F0 - kDiHalo, 0LL), f_hi = min(F0 + kDiF, n);
    const int nq = (nc + 7) >> 3;
    for (int i = threadIdx.x; i < (int)(f_hi - f_lo) * 8; i += kDiThreads) {
        const int q = i & 7;
        if (q >= nq) continue;
        const long long f = f_lo + (i >> 3), row_end = f * S + c0 + nc;
        const long long qs = f * S + c0 + 8 * q;                  // first sample of channels c0 + 8q ..
        const long long sv = qs >> 3;
        const int k = (int)(qs & 7);
        const uint4 lo = ld_nc_v4(src + sv * 8);                  // holds qs, inside the row
        const uint4 hi = k && (sv + 1) * 8 < row_end ? ld_nc_v4(src + (sv + 1) * 8) : make_uint4(0, 0, 0, 0);
        uint32_t o[4];
        realign8(lo, hi, k, o);
#pragma unroll
        for (int e = 0; e < 8; e++) {
            const int c = 8 * q + e;
            if (c >= nc) break;
            const long long p = f - F0 + (sdst[c] & 7);           // destination position in the tile
            if (p >= 0 && p < kDiF) T[di_row(c) * kDiStride + p] = (int16_t)(o[e >> 1] >> (16 * (e & 1)));
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nc * (kDiF / 8); i += kDiThreads) {
        const int j = i % (kDiF / 8), c = i / (kDiF / 8);
        const long long g = sdst[c];
        const long long d0 = ((g >> 3) * 8) + F0 + 8 * j, f0 = d0 - g;   // the vector and its first frame
        if (f0 >= n) continue;
        const uint4 v = *reinterpret_cast<const uint4 *>(T + di_row(c) * kDiStride + 8 * j);
        if (f0 >= 0 && f0 + 8 <= n) {
            *reinterpret_cast<uint4 *>(dst + d0) = v;
        } else {
            const uint32_t o[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < 8; e++)
                if (f0 + e >= 0 && f0 + e < n) dst[d0 + e] = (int16_t)(o[e >> 1] >> (16 * (e & 1)));
        }
    }
}

// samples k .. k + 3 of the eight 32-bit samples in two consecutive aligned vectors
__device__ __forceinline__ void realign4(const uint4 &lo, const uint4 &hi, int k, uint32_t (&o)[4])
{
    const uint32_t w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
#pragma unroll
    for (int t = 0; t < 4; t++) o[t] = k == 0 ? w[t] : k == 1 ? w[t + 1] : k == 2 ? w[t + 2] : w[t + 3];
}

template <typename Tin>
__global__ void __launch_bounds__(kDiThreads) k_stream_frames(const Tin *__restrict__ src, int16_t *__restrict__ dst,
                                                                     const CopySeg *__restrict__ seg, int S, long long n,
                                                                     long long pitch, int e0, int cblocks)
{
    constexpr int V = 16 / sizeof(Tin), L = kDiC / V;             // samples per vector, lanes per row
    constexpr int lgV = V == 8 ? 3 : 2, lgL = V == 8 ? 3 : 4;
    __shared__ __align__(16) int16_t T[kDiC * kDiStride];
    __shared__ long long sdst[kDiC];
    const int c0 = (int)(blockIdx.x % cblocks) * kDiC, nc = min(kDiC, S - c0);
    const long long F0 = (long long)(blockIdx.x / cblocks) * kDiF;
    if (threadIdx.x < nc) sdst[threadIdx.x] = seg[c0 + threadIdx.x].dst;
    __syncthreads();
    const long long f_lo = max(F0 - kDiHalo, 0LL), f_hi = min(F0 + kDiF, n);
    const int nq = (nc + V - 1) / V;
    for (int i = threadIdx.x; i < (int)(f_hi - f_lo) * L; i += kDiThreads) {
        const int q = i & (L - 1);
        if (q >= nq) continue;
        const long long f = f_lo + (i >> lgL), row = e0 + f * pitch + c0, row_end = row + nc;
        const long long qs = row + V * q;                         // first sample of channels c0 + Vq ..
        const long long sv = qs >> lgV;
        const int k = (int)(qs & (V - 1));
        const uint4 lo = ld_nc_v4(src + sv * V);                  // holds qs, inside the row
        const uint4 hi = k && (sv + 1) * V < row_end ? ld_nc_v4(src + (sv + 1) * V) : make_uint4(0, 0, 0, 0);
        uint32_t o[4];
        Tin v[V];
        if constexpr (V == 8) {
            realign8(lo, hi, k, o);
#pragma unroll
            for (int e = 0; e < 8; e++) v[e] = (Tin)(o[e >> 1] >> (16 * (e & 1)));
        } else {
            realign4(lo, hi, k, o);
#pragma unroll
            for (int e = 0; e < 4; e++) memcpy(&v[e], &o[e], 4);
        }
#pragma unroll
        for (int e = 0; e < V; e++) {
            const int c = V * q + e;
            if (c >= nc) break;
            const long long p = f - F0 + (sdst[c] & 7);           // destination position in the tile
            if (p >= 0 && p < kDiF) T[di_row(c) * kDiStride + p] = sample_to_s16(v[e]);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nc * (kDiF / 8); i += kDiThreads) {
        const int j = i % (kDiF / 8), c = i / (kDiF / 8);
        const long long g = sdst[c];
        const long long d0 = ((g >> 3) * 8) + F0 + 8 * j, f0 = d0 - g;   // the vector and its first frame
        if (f0 >= n) continue;
        const uint4 v = *reinterpret_cast<const uint4 *>(T + di_row(c) * kDiStride + 8 * j);
        if (f0 >= 0 && f0 + 8 <= n) {
            *reinterpret_cast<uint4 *>(dst + d0) = v;
        } else {
            const uint32_t o[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < 8; e++)
                if (f0 + e >= 0 && f0 + e < n) dst[d0 + e] = (int16_t)(o[e >> 1] >> (16 * (e & 1)));
        }
    }
}

// Bit windows of open recordings, demodulated as their samples arrive (retention mode AFSK_RETAIN_BITS): job j decides
// windows 0 .. nwin - 1 of one recording range, window k = samples x0 + k bf .. + bf - 1 of the sample arena, into
// plane words w0, w0 + 1, ... of the plane arena.  One lane per window and one ballot per plane word; a CTA takes up to
// kWinTileWords words of one job, so its bit length is uniform and the {mark, space} weights of every 8-sample step of
// a window sit in shared memory (read as a broadcast).  A lane reads its window with aligned 128-bit loads realigned
// to the window start (the window alignment is arbitrary), then the same per-sample arithmetic as k_demod: the
// limiter and template sums of accum4_full in packed accumulators flushed every kFlushVecs vectors, the decision
// with tie_bit, and quiet <=> sum |x| < amp_end * bf.
struct __align__(16) WinJob {
    int64_t x0;          // sample-arena index of window 0's first sample
    int64_t w0;          // plane-arena word of windows 0 .. 31
    int32_t nwin;        // windows to decide (> 0)
    int32_t bf;          // bit length: a multiple of 4, at most kWinMaxBf
    int32_t thr_bf;      // amp_end * bf
    int32_t pad;
};
constexpr int kWinWarps = 4, kWinTileWords = 16, kWinMaxBf = 2000;
constexpr int64_t kBitsMaxPiece = (int64_t)1 << 32;   // frames per channel and push in bits mode (WinJob.nwin < 2^31 at bf = 4)

__global__ void __launch_bounds__(32 * kWinWarps) k_stream_windows(const int16_t *__restrict__ x, uint2 *__restrict__ planes,
                                                                  const WinJob *__restrict__ jobs,
                                                                  const int64_t *__restrict__ tile_first, int n)
{
    __shared__ uint4 wt[kWinMaxBf / 8 + 1];      // step i: {mark, space} of window samples 8i .. 8i + 3, then 8i + 4 .. 8i + 7
    const long long tile = blockIdx.x;
    int a = 0, b = n;                              // job of this tile
    while (b - a > 1) {
        const int mid = (a + b) >> 1;
        if (tile_first[mid] <= tile) a = mid; else b = mid;
    }
    const WinJob J = jobs[a];
    const int bf = J.bf, nvec = (bf + 7) >> 3;
    for (int i = threadIdx.x; i < nvec; i += blockDim.x)
        wt[i] = make_uint4(tone_weights4(bf, 8 * i, false), tone_weights4(bf, 8 * i, true), tone_weights4(bf, 8 * i + 4, false),
                           tone_weights4(bf, 8 * i + 4, true));
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long word0 = (tile - tile_first[a]) * kWinTileWords;
    const long long word1 = min(word0 + kWinTileWords, (long long)((J.nwin + 31) >> 5));
    const uint32_t k512 = 0x02000200u | ((uint32_t)bf >> 16);     // (one register, as in k_demod)
    for (long long wd = word0 + warp; wd < word1; wd += kWinWarps) {
        const long long k = wd * 32 + lane;
        bool bit = false, quiet = false;
        if (k < J.nwin) {
            const long long s0 = J.x0 + k * bf;
            const uint4 *src = reinterpret_cast<const uint4 *>(x) + (s0 >> 3);
            const int sh = (int)(s0 & 7);
            int Um = 0, Nm = 0, Us = 0, Ns = 0, accA = 0;
            uint4 lo = __ldg(src);
            for (int i0 = 0; i0 < nvec; i0 += kFlushVecs) {
                const int i1 = min(nvec, i0 + kFlushVecs);
                int accM = 0, accS = 0;
                for (int i = i0; i < i1; i++) {
                    const uint4 hi = __ldg(src + i + 1);   // (at most one vector past the window: the arena's pad)
                    uint32_t o[4];
                    realign8(lo, hi, sh, o);
                    lo = hi;
                    const uint4 w = wt[i];
                    accum4_full(o[0], o[1], w.x, w.y, k512, accM, accS, accA);
                    if (8 * i + 4 < bf) accum4_full(o[2], o[3], w.z, w.w, k512, accM, accS, accA);
                }
                unpack_acc(accM, Um, Nm);
                unpack_acc(accS, Us, Ns);
            }
            bit = Um > Us || (Um == Us && Ns > Nm && tie_bit(Um, Nm, Ns, bf));
            quiet = accA < J.thr_bf;
        }
        const uint32_t bw = __ballot_sync(0xFFFFFFFFu, bit), qw = __ballot_sync(0xFFFFFFFFu, quiet);
        if (lane == 0) planes[J.w0 + wd] = make_uint2(bw, qw);
    }
}

// Framing of open recordings as their windows are decided (retention mode AFSK_RETAIN_PAYLOAD).  A channel's pending
// recording with a stored clock has a FrameState: training (searching for 1,0,0,0 from window `consumed` on), payload
// (k0 known: searching for the first quiet window from `consumed` on, whole 14-window groups decoded into the channel's
// payload slot) and ended (k1 found: the result is fixed).  Job j frames windows [consumed, k_end) of one recording from
// the state the job carries (the host's copy of the state the last push left); a final job (the recording became final
// with K = k_end windows) then writes its AfskRxResult as k_frame does and copies its payload to out.  A channel can have
// two jobs in one launch (its recording became final and a new one was framed), so no job reads `state`: each only
// writes the state it ends with to state[ch] for the host to read back, and a final job that shares its channel with
// a pending job leaves state[ch] to that job (kFrKeepState), so every slot has at most one writer and no reader.  The
// planes hold only the words from the one of window consumed - 3 (training) or of the next incomplete byte (payload)
// on, so nothing below those is read.
struct __align__(16) FrameState {
    long long consumed;  // windows framed
    long long k0;        // payload / ended: first payload window
    long long k1;        // ended: first quiet window at or after k0
    long long nbytes;    // bytes decoded into the payload slot
    int phase;           // 0 training, 1 payload, 2 ended
    int pad[3];
};
static_assert(sizeof(FrameState) == 48, "FrameState layout");
struct __align__(16) FrameJob {
    FrameState start;    // the recording's state before this job (zero for a recording whose clock was just stored)
    int64_t w0;          // plane-arena word of the recording's windows 0 .. 31 (may lie below the words kept)
    int64_t k_end;       // frame up to this window
    int64_t y0;          // payload-arena byte of the recording's byte 0
    int64_t out_off;     // final: offset of the payload in out
    int32_t ch;          // FrameState of the channel
    int32_t flags;       // kFrFinal, kFrKeepState
    int32_t clk, bf;
    int32_t res;         // final: result index
    int32_t pad[3];
};
constexpr int kFrFinal = 1;       // the recording became final with k_end windows
constexpr int kFrKeepState = 4;   // final: another job of this launch owns the channel's state (else it is reset)
constexpr int kStreamFrameWarps = 4;

// minimum over the warp of a non-negative 64-bit value: the high words first, then the low words of the lanes that hold it
__device__ __forceinline__ long long warp_min64(long long v)
{
    const uint32_t hi = __reduce_min_sync(0xFFFFFFFFu, (uint32_t)((unsigned long long)v >> 32));
    const uint32_t lo = __reduce_min_sync(0xFFFFFFFFu, (uint32_t)((unsigned long long)v >> 32) == hi ? (uint32_t)v : 0xFFFFFFFFu);
    return (long long)(((unsigned long long)hi << 32) | lo);
}

__global__ void __launch_bounds__(32 * kStreamFrameWarps) k_stream_frame(const uint2 *__restrict__ planes, uint8_t *__restrict__ pay,
                                                                        FrameState *__restrict__ state, const FrameJob *__restrict__ jobs,
                                                                        uint8_t *__restrict__ out, AfskRxResult *__restrict__ res, int n)
{
    __shared__ uint8_t lut[128];
    static_assert(32 * kStreamFrameWarps == 128, "one LUT entry per thread");
    const int tid = threadIdx.x, lane = tid & 31;
    lut[tid] = (uint8_t)hamming74_nibble((uint32_t)tid);
    __syncthreads();
    const int j = blockIdx.x * kStreamFrameWarps + (tid >> 5);
    if (j >= n) return;
    const FrameJob J = jobs[j];
    FrameState F = J.start;
    const uint32_t *PW = reinterpret_cast<const uint32_t *>(planes);        // word w: bits PW[2w], quiet PW[2w + 1]
    const long long K = J.k_end;
    constexpr long long NONE = 0x7FFFFFFFFFFFFFFFLL;
    long long c = F.consumed;
    if (F.phase == 0 && c < K) {
        // (:362-366) from window c on; a word's predecessor is read only where its bits enter windows >= c
        long long kt = NONE;
        for (long long base = c >> 5; base <= (K - 1) >> 5; base += 32) {
            const long long w = base + lane;
            long long cand = NONE;
            if (w <= (K - 1) >> 5) {
                const uint32_t cur = PW[2 * (J.w0 + w)];
                const uint32_t prev = (w > 0 && c < 32 * w + 3) ? PW[2 * (J.w0 + w - 1)] : 0u;
                uint32_t M = term_mask(prev, cur);
                if (w == (c >> 5)) M &= ~((1u << (c & 31)) - 1u);
                const long long rem = K - 32 * w;
                if (rem < 32) M &= (1u << rem) - 1u;
                if (M) cand = 32 * w + (__ffs(M) - 1);
            }
            kt = warp_min64(cand);
            if (kt != NONE) break;
        }
        if (kt != NONE) { F.phase = 1; F.k0 = kt + 1; c = F.k0; } else { c = K; }
    }
    if (F.phase == 1) {
        long long kq = NONE;
        if (c < K) {
            // (:372-378) first quiet window at or after c (>= k0)
            for (long long base = c >> 5; base <= (K - 1) >> 5; base += 32) {
                const long long w = base + lane;
                long long cand = NONE;
                if (w <= (K - 1) >> 5) {
                    uint32_t M = PW[2 * (J.w0 + w) + 1];
                    if (w == (c >> 5)) M &= ~((1u << (c & 31)) - 1u);
                    const long long rem = K - 32 * w;
                    if (rem < 32) M &= (1u << rem) - 1u;
                    if (M) cand = 32 * w + (__ffs(M) - 1);
                }
                kq = warp_min64(cand);
                if (kq != NONE) break;
            }
        }
        if (kq != NONE) { F.phase = 2; F.k1 = kq; }
        c = max(c, K);
        const long long lim = kq != NONE ? kq : c;                // decoded bytes end before window lim
        // whole 14-window groups (:393-399), one byte per lane
        const long long nb = (lim - F.k0) / 14;
        for (long long i = F.nbytes + lane; i < nb; i += 32) {
            const long long pos = F.k0 + 14 * i;
            const uint32_t lo = PW[2 * (J.w0 + (pos >> 5))], hi = PW[2 * (J.w0 + (pos >> 5) + 1)];
            pay[J.y0 + i] = (uint8_t)decode_byte(__funnelshift_r(lo, hi, (uint32_t)(pos & 31)) & 0x3FFFu, lut);
        }
        F.nbytes = max(F.nbytes, nb);
    }
    F.consumed = max(F.consumed, c);
    if (J.flags & kFrFinal) {
        const long long k0 = F.phase >= 1 ? F.k0 : K, k1 = F.phase == 2 ? F.k1 : K;
        const long long nbits = k1 - k0;
        __syncwarp();                                            // the bytes decoded above, read back by other lanes
        for (long long i = lane; i < F.nbytes; i += 32) out[J.out_off + i] = pay[J.y0 + i];
        if (lane == 0) {
            AfskRxResult r;
            r.status = nbits > 0 ? AFSK_ST_OK : AFSK_ST_NO_DATA;
            r.clock = J.clk;
            r.train_end = (long long)J.clk + k0 * J.bf;          // "Training sequence terminated on frame" :368
            r.nbits = nbits;
            r.nbytes = nbits > 0 ? F.nbytes : 0;
            res[J.res] = r;
            if (!(J.flags & kFrKeepState)) state[J.ch] = FrameState{0, 0, 0, 0, 0, {0, 0, 0}};
        }
    } else if (lane == 0) {
        state[J.ch] = F;
    }
}

struct Group {
    int bf = 0, tpw_log2 = 0, seg = 0, nv = 0, nt = 0, merge = 0, wt = 0, nsub = 1, stage_bytes = 0, stages = 0;
    int small_wpt = 0;            // > 0: k_demod_lane<bf/8, small_wpt>
    int shift_wpt = 0;            // > 0: k_demod_shift<bf, shift_wpt>
    int pad = 0;                  // 1: padded layout, k_demod_shift<bf, shift_wpt, true> (cp.async producer)
    size_t smem = 0;
    int grid = 0;
    // fused mode (auxiliary warps): shared memory with the AuxSmem block appended, its offset, the grid for
    // that footprint, the exact multiply-shift for floor(D / 2bf), per-capture arrival counters and job counters
    size_t smem_fused = 0;
    int aux_off = 0, grid_fused = 0;
    bool can_fuse = false;
    uint32_t clk_magic = 0;
    int clk_shift = 0;
    std::vector<int32_t> caps, tile_first, tile_gpos;
    int32_t *d_caps = nullptr, *d_tile_first = nullptr, *d_tile_gpos = nullptr;   // inside the plan's arena
    uint32_t *d_tiles_done = nullptr, *d_ctrl = nullptr;
};

}  // namespace

// kernel variants: merge mode with 1..6 vector steps, plain mode with 2..7, generic fallback
#define AFSK_DEMOD_VARIANTS(X) \
    X(1, true) X(2, true) X(3, true) X(4, true) X(5, true) X(6, true) \
    X(2, false) X(3, false) X(4, false) X(5, false) X(6, false) X(7, false) X(0, false)

// k_demod_shift instantiations: (bit length, windows per thread)
#define AFSK_SHIFT_VARIANTS(X) X(4, 8) X(12, 4) X(20, 2) X(60, 2) X(100, 2) X(120, 1) X(200, 1)
// the same with the padded layout (thread segments of 16 vectors)
#define AFSK_PAD_VARIANTS(X) X(32, 4) X(64, 2) X(128, 1)

static cudaError_t demod_set_smem_attr()
{
    cudaError_t e = cudaFuncSetAttribute(k_demod_lane<1, 8, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
#define X(BF, W) \
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_demod_shift<BF, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    AFSK_SHIFT_VARIANTS(X)
#undef X
#define X(BF, W) \
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_demod_shift<BF, W, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    AFSK_PAD_VARIANTS(X)
#undef X
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_demod_lane<2, 4, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_demod_lane<3, 2, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
#define X(NT, MG) \
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_demod<NT, MG>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    AFSK_DEMOD_VARIANTS(X)
#undef X
    return e;
}

static void launch_demod(int merge, int nt, int grid, int block, size_t smem, cudaStream_t st, const DemodParams &p)
{
#define X(NT, MG) \
    if ((MG) == (merge != 0) && (NT) == nt) { k_demod<NT, MG><<<grid, block, smem, st>>>(p); return; }
    AFSK_DEMOD_VARIANTS(X)
#undef X
    DemodParams q = p;          // no specialised variant: generic loop over nv vectors
    q.merge = 0;
    k_demod<0, false><<<grid, block, smem, st>>>(q);
}

// the kernel a group is demodulated with (same selection as the launch), for occupancy queries
static const void *demod_kernel_of(const Group &g)
{
    if (g.small_wpt && g.bf == 8) return (const void *)k_demod_lane<1, 8, 8>;
    if (g.small_wpt && g.bf == 16) return (const void *)k_demod_lane<2, 4, 8>;
    if (g.small_wpt && g.bf == 24) return (const void *)k_demod_lane<3, 2, 8>;
#define X(BF, W) \
    if (g.pad && g.shift_wpt == (W) && g.bf == (BF)) return (const void *)k_demod_shift<BF, W, true>;
    AFSK_PAD_VARIANTS(X)
#undef X
#define X(BF, W) \
    if (!g.pad && g.shift_wpt == (W) && g.bf == (BF)) return (const void *)k_demod_shift<BF, W>;
    AFSK_SHIFT_VARIANTS(X)
#undef X
#define X(NT, MG) \
    if ((MG) == (g.merge != 0) && (NT) == g.nt) return (const void *)k_demod<NT, MG>;
    AFSK_DEMOD_VARIANTS(X)
#undef X
    return (const void *)k_demod<0, false>;
}

struct AfskRxPlan {
    int device = 0;
    int B = 0;
    int sm_count = 148;
    std::vector<CapDesc> caps;
    std::vector<int64_t> out_off;
    std::vector<Group> groups;
    // ONE device allocation (grow-only, reused by afsk_rx_plan_reset): descriptor block (capture
    // descriptors, then every group's capture list / tile prefix / tile map), clock indices, bit planes
    uint8_t *arena = nullptr;
    size_t arena_bytes = 0;
    std::vector<uint8_t> h_desc;  // host image of the descriptor block: one H2D copy per (re)build
    CapDesc *d_caps = nullptr;
    int32_t *d_clock = nullptr;
    uint2 *d_planes = nullptr;
    int64_t plane_words = 0;
    int64_t max_windows = 0;
    int64_t sum_windows = 0;      // over the captures decoded on the GPU
    int64_t gpu_caps = 0;
    unsigned long long *d_cready = nullptr;   // fused mode: {clock, epoch tag} per capture
    uint32_t epoch = 0;           // decodes issued with this plan (fused mode tags)
    int n_preset = 0;             // captures whose result is decided on the host (status0 != 0)
    int64_t sum_samples = 0;      // over the captures decoded on the GPU
    bool can_fuse = false;        // every group fits the auxiliary warps (bit length, shared memory)
    int fused = -1;               // AFSK_OPT_FUSED: -1 automatic, 0 three kernels, 1 fused clocks, 2 fused clocks and framing
    int clock_kernel = 0;         // AFSK_OPT_CLOCK_KERNEL: 0 automatic (k_clock_q for bit lengths 8..24, k_clock for the rest), 1 k_clock, 2 k_clock2 (bit lengths up to kAuxMaxBf)
    bool can_clock2 = false;
    int frame_kernel = 0;         // AFSK_OPT_FRAME_KERNEL: 0 automatic, 1 k_frame_warp, 2 k_frame<128,4,int>, 3 <512,8,int>, 4 <512,8,long long>
    int l2_hint = -1;             // AFSK_OPT_L2_HINT / AFSK_L2_HINT (read once per plan): -1 per-kernel default
    bool timing = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timing_events;
    int timed_launches = 0;       // demodulator launches covered by timing_events
    // one stream per baud group after the first: the groups' kernels are independent (disjoint captures), so the
    // next group's CTAs fill the SMs as the previous group's drain instead of waiting for its last CTA
    int rot = 1;                  // rotated vector order at 32-sample segments (tuning switch AFSK_NO_ROT)
    int group_streams = 1;        // AFSK_OPT_GROUP_STREAMS
    int pad_warps = 0;            // padded layout: producer warps per CTA, 0 = per group (tuning switch AFSK_PAD_WARPS, read at plan creation)
    std::vector<cudaStream_t> gstreams;
    std::vector<cudaEvent_t> gevents;   // [0] fork, [i] join of group i
};

// shared-memory ring of two CTAs per SM (228 KB per SM, 1 KB reserved per CTA).  Measured in one
// process on config 2 (tools/ab_demod.py): 2 stages 6204 GB/s, 3 stages 6760, 4 stages 6690, 5 stages
// 6513 — deeper rings do not help once the consumers keep up, so three it is (AFSK_DEMOD_STAGES
// overrides, for tuning runs).
constexpr size_t kDemodSmemBudget = 108 * 1024;
constexpr size_t kDemodMaxStages = 3;

static size_t demod_smem_bytes(const Group &g)
{
    if (g.shift_wpt || g.small_wpt)
        return (size_t)g.stages * g.stage_bytes + kMaxStages * sizeof(TileMeta) + 2 * kMaxStages * sizeof(uint64_t);
    return (size_t)g.stages * g.stage_bytes + (size_t)(1 << g.tpw_log2) * (8 * (2 * g.nt + 1) + 1) * 16 +
           kMaxStages * sizeof(TileMeta) + 2 * kMaxStages * sizeof(uint64_t) + 2 * kConsumerThreads;
}

static int pick_stages(int stage_bytes)
{
    const size_t fit = std::max<size_t>(1, kDemodSmemBudget / (size_t)stage_bytes);
    size_t want = kDemodMaxStages;
    const char *ev = getenv("AFSK_DEMOD_STAGES");
    if (ev && atoi(ev) > 0) want = (size_t)atoi(ev);
    return (int)std::min<size_t>(std::min<size_t>(want, fit), kMaxStages);
}

static bool configure_group(Group &g, int bf)
{
    g.bf = bf;
    g.tpw_log2 = 0;
    if (bf == 8 || bf == 16 || bf == 24) {
        // short windows: lane-major tiles of 256 * kJ windows (k_demod_lane<bf/8, kJ, 8 warps>), kJ = 8 / 4 / 2.  Smaller
        // tiles are slower (6000 baud, same box: 32 KB tiles 6661 GB/s, 16 KB 5756-6079, 8 KB 4715)
        g.small_wpt = bf == 8 ? 8 : (bf == 16 ? 4 : 2);
        // (48 KB tiles in a two-stage ring, kJ = 12 / 6 / 3: 6000 baud 6570 -> 6485 GB/s, 3000 baud 6783 -> 6844, 2000 baud
        // 6789 -> 6877 on one box: not worth the extra instantiations)
        g.seg = bf * g.small_wpt;
        g.nv = g.seg / 8 + 1;
        g.nt = g.nv; g.merge = 0;
        g.wt = kConsumerThreads * g.small_wpt;
        g.stage_bytes = ((g.wt * bf * 2 + 16 + 256) + 127) & ~127;
        g.stages = pick_stages(g.stage_bytes);
        g.smem = demod_smem_bytes(g);
        return true;
    }
    // 800 / 480 / 400 / 240 baud (60 / 100 / 120 / 200 samples per bit): in the general kernel a thread's segment is not a whole
    // number of vectors there (masked head / tail vectors, weight table in shared memory: 4.8 / 4.0 / 4.6 / 3.4 TB/s);
    // k_demod_shift with 2 / 2 / 1 / 1 windows per thread reads 15 or 25 whole vectors per thread, conflict-free (odd
    // multiples of 16 bytes between threads): 6.8 / 7.0 / 7.0 / 6.9 TB/s.  (The same kernel at 1200 / 1000 / 500 baud:
    // 5.6 TB/s against 6.9 / 6.9 / 6.5 of the general kernel; at 600 / 300 baud within 1 %: they stay where they are.)
    const bool long_shift = (bf == 60 || bf == 100 || bf == 120 || bf == 200) && !getenv("AFSK_NO_LONG_SHIFT");
    if (bf == 4 || bf == 12 || bf == 20 || long_shift) {
        // windows whose thread segment is not a whole number of vectors in the general kernel: k_demod_shift with as many
        // windows per thread as make it one (4000 / 2400 baud: 4 / 2 windows; 800 / 480 baud: 2; 400 / 240 baud: 1 window of
        // 15 / 25 vectors).  The long ones are 60-100 KB per tile: one CTA per SM with a 2-3 stage ring.
        g.shift_wpt = bf == 4 ? 8 : (bf == 12 ? 4 : ((bf == 20 || bf == 60 || bf == 100) ? 2 : 1));   // 12000 baud: eight 4-sample windows per thread   // measured at 4000 baud: 4 windows per thread 6245 GB/s, 2 -> 5366
        g.seg = bf * g.shift_wpt;
        g.nv = g.seg / 8 + 1;
        g.nt = g.nv; g.merge = 0;
        g.nsub = long_shift ? 1 : 2;         // two sub-tiles per tile: 4000 baud 5932 -> 6178 GB/s, 2400 baud 6006 -> 6397 (same box)
        if (const char *ev = getenv("AFSK_DEMOD_NSUB")) g.nsub = std::max(1, std::min(8, atoi(ev)));
        g.wt = g.nsub * kConsumerThreads * g.shift_wpt;
        g.stage_bytes = ((g.wt * bf * 2 + 16 + 256) + 127) & ~127;
        g.stages = pick_stages(g.stage_bytes);
        if (long_shift) g.stages = (int)std::min<size_t>(3, (size_t)(220 * 1024) / (size_t)g.stage_bytes);
        g.smem = demod_smem_bytes(g);
        // a ring needs one stage: a tile larger than the budget (AFSK_DEMOD_NSUB=3 at 480 / 240 baud, ~307 KB) is refused
        return g.stages >= 1;
    }
    if ((bf == 32 || bf == 64 || bf == 128) && !getenv("AFSK_NO_PAD")) {
        // 1500 / 750 / 375 baud: power-of-two windows.  Four / two / one windows per thread over the padded layout
        // (demod_produce_pad): 16 vectors per thread segment and one spare vector after each (stride 17 vectors: conflict-free
        // 128-bit reads).  Tiles of 70 KB in a 3-stage ring, one CTA per SM, like the long k_demod_shift windows.
        // Same box, general kernel -> padded: 1500 baud 4994 -> 5901 GB/s, 750 baud 4147 -> 5906, 375 baud 4050 -> 6328;
        // segments of 8 -> 16 vectors at 1500 / 750 baud (37 KB tiles, two CTAs per SM before): 5811 -> 6120 and 5717 -> 6232
        // (the per-window epilogue and the per-thread head / tail handling are shared by twice the samples).
        // (Measured and rejected: the same layout at 300 / 600 / 4000 baud, 5908 / 5795 / 6364 against 6210 / 6277 / 6357.)
        g.shift_wpt = 128 / bf;
        g.pad = 1;
        g.seg = bf * g.shift_wpt;
        g.nv = g.seg / 8 + 1;
        g.nt = g.nv; g.merge = 0;
        g.nsub = 1;
        if (const char *ev = getenv("AFSK_DEMOD_NSUB")) g.nsub = std::max(1, std::min(8, atoi(ev)));
        g.wt = g.nsub * kConsumerThreads * g.shift_wpt;
        g.stage_bytes = (((8 + g.nsub * kConsumerThreads * (g.seg / 8 + 1) + 2) * 16) + 127) & ~127;
        g.stages = (int)std::min<size_t>(3, (size_t)(220 * 1024) / (size_t)g.stage_bytes);
        if (const char *ev = getenv("AFSK_DEMOD_STAGES")) g.stages = std::max(1, std::min(kMaxStages, atoi(ev)));
        g.smem = demod_smem_bytes(g);
        return g.stages >= 1 && g.smem <= 227 * 1024;
    }
    // Segments of at most 48 samples per thread.  The thread stride in shared memory is 2 * seg bytes:
    // 40 samples (80 B) is conflict-free for 128-bit loads and 48 is 2-way, both reach the HBM ceiling;
    // 32 is 4-way (75-89 % of it: 1500 / 750 / 375 baud).  Measured and rejected: segments of 64
    // samples in merge mode (8-way, 57 %) and two 32-sample windows per thread (83 %).
    while ((bf >> g.tpw_log2) > 48 && g.tpw_log2 < 3) g.tpw_log2++;
    // Two sub-tiles per tile (three where a thread's segment is 32 samples): 40-48 KB tiles in a 2-stage ring
    // instead of 16-24 KB tiles in a 3-stage ring.  Same box, alternating runs (gpurun_out/r2e, r2e2; GB/s of the
    // demodulator): 1200 baud 6600 -> 6880, 300 baud 5820 -> 6130, 1000 baud 6786 -> 6935, 500 baud 6069 -> 6350,
    // 800 baud 4533 -> 4765, 480 baud 3766 -> 3974, 400 baud 4398 -> 4603, 240 baud 3219 -> 3431; 1500 / 750 / 375 baud
    // 5814 / 5031 / 4565 -> 5813 / 5371 / 4854 with three.  Three sub-tiles elsewhere cost a ring stage (c2: 5937).
    // (Shorter segments with more threads per window, to halve the bank conflicts of 32-sample segments, lose far
    // more in shuffles than they gain: 1500 baud 4124 GB/s.)
    g.nsub = (bf == 32 || bf == 64 || bf == 128) ? 3 : 2;
    if (const char *ev = getenv("AFSK_DEMOD_TPW_LOG2")) g.tpw_log2 = std::max(0, std::min(3, atoi(ev)));   // tuning runs
    if (const char *ev = getenv("AFSK_DEMOD_NSUB")) g.nsub = std::max(1, std::min(8, atoi(ev)));
    const int tpw = 1 << g.tpw_log2;
    g.seg = (bf + tpw - 1) / tpw;
    g.nv = (g.seg + 6) / 8 + 1;
    g.merge = (g.seg % 8 == 0 && g.seg <= 48 && bf % tpw == 0) ? 1 : 0;   // then bf == tpw * seg and nv == seg/8 + 1
    g.nt = g.merge ? g.nv - 1 : g.nv;
    // (one CTA per SM with 60-80 KB tiles, which is what suits k_demod_shift's long per-thread segments, loses here:
    //  1200 baud 5980 GB/s, 300 baud 4970, 600 baud 5250)
    for (;; g.nsub--) {
        g.wt = g.nsub * (kConsumerThreads / tpw);
        g.stage_bytes = ((g.wt * bf * 2 + g.nv * 16 + 2 * tpw + 256) + 127) & ~127;   // copy (e0 < 64) + over-read slack
        g.stages = pick_stages(g.stage_bytes);
        g.smem = demod_smem_bytes(g);
        while (g.smem > 113 * 1024 && g.stages > 2) {      // keep two CTAs per SM when the tables are large
            g.stages--;
            g.smem = demod_smem_bytes(g);
        }
        // very long bits (below 100 baud): the sub-tiled ring would not leave two stages and two CTAs per SM
        if (g.nsub == 1 || (g.smem <= 113 * 1024 && g.stages >= 2)) break;
    }
    while (g.smem > 227 * 1024 && g.stages > 1) {
        g.stages--;
        g.smem = demod_smem_bytes(g);
    }
    return g.smem <= 227 * 1024;
}

// scratch of one gate call: freed on every exit path
struct GateScratch {
    int64_t *d_first = nullptr, *d_off = nullptr;
    int32_t *d_amp = nullptr;
    ~GateScratch() { cudaFree(d_first); cudaFree(d_off); cudaFree(d_amp); }
};

// chunk amplitudes of S streams, then one open/close search (max_calls < 0, k_gate_scan) or the walk
// of successive receive() calls (k_gate_multi)
static int gate_run(int device, const int16_t *d_samples, const int64_t *h_offsets, int S, int amp_start, int amp_end,
                    int64_t timeout_frames, int max_calls, int64_t *d_ranges, int32_t *d_counts, void *stream)
{
    if (S == 0) return AFSK_OK;
    if ((reinterpret_cast<uintptr_t>(d_samples) & 15) != 0) { afsk_set_error("gate: d_samples must be 16-byte aligned"); return AFSK_E_ARG; }
    AfskDeviceGuard guard(device);
    if (!guard.ok) { afsk_set_error("cannot select device %d", device); return AFSK_E_CUDA; }
    cudaStream_t st = (cudaStream_t)stream;
    std::vector<int64_t> first((size_t)S + 1, 0);
    for (int s = 0; s < S; s++) {
        if (h_offsets[s + 1] < h_offsets[s] || h_offsets[s] < 0) { afsk_set_error("gate: offsets must be non-negative and non-decreasing"); return AFSK_E_ARG; }
        first[s + 1] = first[s] + (h_offsets[s + 1] - h_offsets[s]) / AFSK_GATE_CHUNK;
    }
    const long long total = first[S];
    GateScratch g;
    AFSK_CUDA(cudaMalloc((void **)&g.d_first, sizeof(int64_t) * ((size_t)S + 1)));
    AFSK_CUDA(cudaMalloc((void **)&g.d_off, sizeof(int64_t) * ((size_t)S + 1)));
    AFSK_CUDA(cudaMalloc((void **)&g.d_amp, sizeof(int32_t) * (size_t)(total ? total : 1)));
    AFSK_CUDA(cudaMemcpyAsync(g.d_first, first.data(), sizeof(int64_t) * ((size_t)S + 1), cudaMemcpyHostToDevice, st));
    AFSK_CUDA(cudaMemcpyAsync(g.d_off, h_offsets, sizeof(int64_t) * ((size_t)S + 1), cudaMemcpyHostToDevice, st));
    if (total > 0) {
        const int wpb = 8;
        k_gate_amp<<<(unsigned)((total + wpb - 1) / wpb), wpb * 32, 0, st>>>(d_samples, g.d_first, g.d_off, S, total, g.d_amp);
    }
    if (max_calls < 0) k_gate_scan<<<S, kFrameThreads, 0, st>>>(g.d_amp, g.d_first, amp_start, amp_end, timeout_frames, d_ranges);
    else k_gate_multi<<<S, 32, 0, st>>>(g.d_amp, g.d_first, GateParams{amp_start, amp_end, timeout_frames}, nullptr, max_calls,
                                         nullptr, 1, nullptr, nullptr, d_ranges, d_counts);
    AFSK_CUDA(cudaGetLastError());
    AFSK_CUDA(cudaStreamSynchronize(st));     // the host staging vector and the scratch go out of scope
    return AFSK_OK;
}

// (Re)builds every host- and device-side descriptor of a plan for a batch layout.  The device arena is
// reused when it is large enough (grow-only), so re-targeting a plan costs one H2D copy of the
// descriptor block and no allocation.
static int plan_build(AfskRxPlan *P, int B, const int64_t *h_start, const int64_t *h_len, const int32_t *h_baud,
                      const int32_t *h_amp_end)
{
    P->B = B;
    P->caps.assign((size_t)B, CapDesc());
    P->out_off.assign((size_t)B + 1, 0);
    P->groups.clear();
    P->max_windows = P->sum_windows = P->gpu_caps = P->sum_samples = 0;
    P->n_preset = 0;
    std::map<int, int> bf_to_group;
    int64_t words = 0;
    for (int c = 0; c < B; c++) {
        CapDesc &d = P->caps[c];
        d.off = h_start[c];
        d.n = h_len[c];
        if (d.n < 0 || d.off < 0) { afsk_set_error("capture %d: negative start or length (offsets must be non-decreasing)", c); return AFSK_E_ARG; }
        d.plane_base = words;
        d.out_off = P->out_off[c];
        d.group = -1;
        int bf = 0, ml = 0, sl = 0;
        long long thr = h_amp_end[c];
        d.thr = (int32_t)std::min<long long>(std::max<long long>(thr, 0), 65537);
        if (!afsk_tone_geometry(h_baud[c], &bf, &ml, &sl)) {
            d.bf = 0; d.status0 = AFSK_ST_EXC_BAUD;
        } else {
            d.bf = bf;
            if (d.n < AFSK_SYNC_FRAMES) d.status0 = AFSK_ST_NO_CLOCK;                 // :323-325
            else if (AFSK_SYNC_FRAMES - 2 * bf <= 0) d.status0 = AFSK_ST_EXC_INDEX;   // :332 on []
            else if (ml != bf || sl != bf) d.status0 = AFSK_ST_EXC_WAVELEN;           // :102-103
            else d.status0 = 0;
        }
        int64_t cap_bytes = 16;
        if (d.status0 == 0) {
            auto it = bf_to_group.find(bf);
            if (it == bf_to_group.end()) {
                Group g;
                if (!configure_group(g, bf)) { afsk_set_error("bit_frames %d needs too much shared memory", bf); return AFSK_E_UNSUPPORTED; }
                g.tile_first.push_back(0);
                P->groups.push_back(g);
                it = bf_to_group.emplace(bf, (int)P->groups.size() - 1).first;
            }
            Group &g = P->groups[it->second];
            d.group = it->second;
            const int64_t kmax = (d.n - bf + bf - 1) / bf;             // windows at clock 0
            const int64_t ntiles = (kmax + g.wt - 1) / g.wt;
            P->max_windows = std::max(P->max_windows, kmax);
            P->sum_windows += kmax;
            P->sum_samples += d.n;
            P->gpu_caps++;
            if (ntiles + (int64_t)g.tile_first.back() > 0x7FFFFFF0LL) { afsk_set_error("batch too large"); return AFSK_E_ARG; }
            g.caps.push_back(c);
            g.tile_gpos.insert(g.tile_gpos.end(), (size_t)ntiles, (int32_t)g.caps.size() - 1);
            g.tile_first.push_back(g.tile_first.back() + (int32_t)ntiles);
            words += ntiles * (g.wt / 32) + 4;
            cap_bytes = (kmax / 14 + 16 + 15) & ~(int64_t)15;
        } else {
            P->n_preset++;
        }
        P->out_off[c + 1] = P->out_off[c] + cap_bytes;
    }
    P->plane_words = words + 8;

    // ---- descriptor block image (every sub-array 16-byte aligned) ----
    auto align16 = [](size_t v) { return (v + 15) & ~(size_t)15; };
    size_t desc_bytes = align16(sizeof(CapDesc) * (size_t)B);
    std::vector<size_t> goff;
    for (Group &g : P->groups) {
        goff.push_back(desc_bytes); desc_bytes += align16(sizeof(int32_t) * g.caps.size());
        goff.push_back(desc_bytes); desc_bytes += align16(sizeof(int32_t) * g.tile_first.size());
        goff.push_back(desc_bytes); desc_bytes += align16(sizeof(int32_t) * g.tile_gpos.size());
        goff.push_back(desc_bytes); desc_bytes += align16(sizeof(uint32_t) * g.caps.size());    // tiles_done: zeros
        goff.push_back(desc_bytes); desc_bytes += align16(sizeof(uint32_t) * 8);                // ctrl[2][4]: zeros
    }
    desc_bytes = (desc_bytes + 255) & ~(size_t)255;
    const size_t clock_off = desc_bytes;
    const size_t cready_off = clock_off + ((sizeof(int32_t) * (size_t)(B ? B : 1) + 255) & ~(size_t)255);
    const size_t planes_off = cready_off + ((sizeof(unsigned long long) * (size_t)(B ? B : 1) + 255) & ~(size_t)255);
    const size_t need = planes_off + sizeof(uint2) * (size_t)P->plane_words;
    P->h_desc.assign(desc_bytes, 0);
    if (B) memcpy(P->h_desc.data(), P->caps.data(), sizeof(CapDesc) * (size_t)B);
    for (size_t gi = 0; gi < P->groups.size(); gi++) {
        Group &g = P->groups[gi];
        memcpy(P->h_desc.data() + goff[5 * gi], g.caps.data(), sizeof(int32_t) * g.caps.size());
        memcpy(P->h_desc.data() + goff[5 * gi + 1], g.tile_first.data(), sizeof(int32_t) * g.tile_first.size());
        memcpy(P->h_desc.data() + goff[5 * gi + 2], g.tile_gpos.data(), sizeof(int32_t) * g.tile_gpos.size());
        g.tile_gpos.clear(); g.tile_gpos.shrink_to_fit();
    }
    cudaError_t e = cudaSuccess;
    if (need > P->arena_bytes) {
        const bool regrow = P->arena != nullptr;
        if (P->arena) cudaFree(P->arena);
        P->arena = nullptr;
        P->arena_bytes = 0;
        const size_t want = regrow ? need + need / 4 : need;        // a plan that is being re-targeted: head-room for the next layout
        e = cudaMalloc((void **)&P->arena, want);
        if (e == cudaSuccess) {
            P->arena_bytes = want;
            // k_frame may load (and mask / shift out) plane words past a capture's last window: keep them
            // defined.  Stale words of an earlier layout are as good as zeros for that purpose.
            e = cudaMemsetAsync(P->arena, 0, want, 0);
        }
    }
    if (e == cudaSuccess && desc_bytes) e = cudaMemcpyAsync(P->arena, P->h_desc.data(), desc_bytes, cudaMemcpyHostToDevice, 0);
    if (e == cudaSuccess) {
        P->d_caps = reinterpret_cast<CapDesc *>(P->arena);
        P->d_clock = reinterpret_cast<int32_t *>(P->arena + clock_off);
        P->d_cready = reinterpret_cast<unsigned long long *>(P->arena + cready_off);
        P->d_planes = reinterpret_cast<uint2 *>(P->arena + planes_off);
        P->can_fuse = !P->groups.empty();
        P->can_clock2 = true;
        for (const Group &g : P->groups) if (g.bf > kAuxMaxBf) P->can_clock2 = false;
        for (size_t gi = 0; gi < P->groups.size(); gi++) {
            Group &g = P->groups[gi];
            g.d_caps = reinterpret_cast<int32_t *>(P->arena + goff[5 * gi]);
            g.d_tile_first = reinterpret_cast<int32_t *>(P->arena + goff[5 * gi + 1]);
            g.d_tile_gpos = reinterpret_cast<int32_t *>(P->arena + goff[5 * gi + 2]);
            g.d_tiles_done = reinterpret_cast<uint32_t *>(P->arena + goff[5 * gi + 3]);
            g.d_ctrl = reinterpret_cast<uint32_t *>(P->arena + goff[5 * gi + 4]);
            const int total = g.tile_first.back();
            // two CTAs per SM even where three would fit: measured on one box, 3 CTAs per SM give 6223 GB/s
            // against 7115 at 1200 baud and 5663 against 6610 at 300 baud (profiles/r1_tuning_log.md)
            const int per_sm = g.smem <= 113 * 1024 ? 2 : 1;
            g.grid = std::max(1, std::min(total, P->sm_count * per_sm));
            // fused mode: the AuxSmem block behind everything else; the CTAs per SM must not drop
            g.aux_off = (int)((g.smem + 15) & ~(size_t)15);
            g.smem_fused = (size_t)g.aux_off + sizeof(AuxSmem);
            const int per_sm_f = g.smem_fused <= 113 * 1024 ? 2 : 1;
            // (the padded-layout kernel's auxiliary warps share the copies of every tile: no fused schedule there)
            g.can_fuse = g.bf <= kAuxMaxBf && g.smem_fused <= 227 * 1024 && per_sm_f == per_sm && !g.pad;
            g.grid_fused = std::max(1, std::min(total, P->sm_count * per_sm_f));
            // floor(D / d) == (D * magic) >> shift for every D < 2^28, d = 2 bf (Granlund-Montgomery: l = ceil(log2 d),
            // magic = ceil(2^(28 + l) / d) < 2^29)
            const uint32_t dv = 2u * (uint32_t)g.bf;
            int l = 0;
            while ((1u << l) < dv) l++;
            g.clk_shift = 28 + l;
            g.clk_magic = (uint32_t)((((unsigned long long)1 << g.clk_shift) + dv - 1) / dv);
            if (!g.can_fuse) P->can_fuse = false;
        }
        static bool attr_set[64] = {};
        if (P->device < 0 || P->device >= 64 || !attr_set[P->device]) {
            e = demod_set_smem_attr();
            if (e == cudaSuccess && P->device >= 0 && P->device < 64) attr_set[P->device] = true;
        }
        // Fused framing waits for other CTAs of the launch: every CTA must be resident.  Ask the runtime how many
        // CTAs of the group's kernel an SM really holds (registers, threads, shared memory) and size the grid to it.
        for (size_t gi = 0; gi < P->groups.size() && e == cudaSuccess; gi++) {
            Group &g = P->groups[gi];
            if (!g.can_fuse) continue;
            const int block = (g.small_wpt || g.shift_wpt) ? kFusedThreads4 : kFusedThreads2;
            int nb = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, demod_kernel_of(g), block, g.smem_fused) != cudaSuccess) nb = 0;
            (void)cudaGetLastError();
            const int per_sm_f = std::min(nb, g.smem_fused <= 113 * 1024 ? 2 : 1);
            if (per_sm_f < 1) { g.can_fuse = false; P->can_fuse = false; continue; }
            g.grid_fused = std::max(1, std::min((int)g.tile_first.back(), P->sm_count * per_sm_f));
        }
    }
    // the set-up ran on the legacy default stream; decodes may use non-blocking streams
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    if (e != cudaSuccess) { afsk_set_error("afsk_rx_plan: %s", cudaGetErrorString(e)); return AFSK_E_CUDA; }
    return AFSK_OK;
}

extern "C" {

int64_t afsk_rx_out_capacity(int64_t n_samples, int baud)
{
    int bf, ml, sl;
    if (n_samples <= 0 || !afsk_tone_geometry(baud, &bf, &ml, &sl)) return 16;
    return (n_samples / bf) / 14 + 16;
}

int afsk_rx_plan_create(int device, int B, const int64_t *h_offsets, const int32_t *h_baud,
                        const int32_t *h_amp_end, AfskRxPlan **plan_out)
{
    if (!plan_out || B < 0 || (B > 0 && (!h_offsets || !h_baud || !h_amp_end))) {
        afsk_set_error("afsk_rx_plan_create: bad argument");
        return AFSK_E_ARG;
    }
    std::vector<int64_t> len((size_t)(B > 0 ? B : 0));
    for (int c = 0; c < B; c++) len[c] = h_offsets[c + 1] - h_offsets[c];
    return afsk_rx_plan_create_ranges(device, B, h_offsets, len.data(), h_baud, h_amp_end, plan_out);
}

int afsk_rx_plan_create_ranges(int device, int B, const int64_t *h_start, const int64_t *h_len, const int32_t *h_baud,
                               const int32_t *h_amp_end, AfskRxPlan **plan_out)
{
    if (!plan_out || B < 0 || (B > 0 && (!h_start || !h_len || !h_baud || !h_amp_end))) {
        afsk_set_error("afsk_rx_plan_create_ranges: bad argument");
        return AFSK_E_ARG;
    }
    AfskDeviceGuard guard(device);
    if (!guard.ok) { afsk_set_error("cannot select device %d", device); return AFSK_E_CUDA; }
    AfskRxPlan *P = new (std::nothrow) AfskRxPlan();
    if (!P) return AFSK_E_ARG;
    P->device = device;
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) P->sm_count = sms;
    const char *ev = getenv("AFSK_L2_HINT");            // tuning overrides, read once per plan
    if (ev) P->l2_hint = atoi(ev);
    ev = getenv("AFSK_FUSED");
    if (ev) P->fused = atoi(ev) < 0 ? -1 : std::min(atoi(ev), 2);
    if (getenv("AFSK_NO_ROT")) P->rot = 0;
    ev = getenv("AFSK_GROUP_STREAMS");
    if (ev) P->group_streams = atoi(ev) ? 1 : 0;
    ev = getenv("AFSK_PAD_WARPS");
    if (ev) P->pad_warps = std::max(1, std::min(5, atoi(ev)));
    ev = getenv("AFSK_CLOCK_KERNEL");
    if (ev && atoi(ev) >= 0 && atoi(ev) <= 2) P->clock_kernel = atoi(ev);
    ev = getenv("AFSK_FRAME_KERNEL");
    if (ev && atoi(ev) >= 0 && atoi(ev) <= 4) P->frame_kernel = atoi(ev);
    const int rc = plan_build(P, B, h_start, h_len, h_baud, h_amp_end);
    if (rc != AFSK_OK) { afsk_rx_plan_destroy(P); return rc; }
    *plan_out = P;
    return AFSK_OK;
}

int afsk_rx_plan_reset(AfskRxPlan *P, int B, const int64_t *h_start, const int64_t *h_len, const int32_t *h_baud,
                       const int32_t *h_amp_end)
{
    if (!P || B < 0 || (B > 0 && (!h_start || !h_baud || !h_amp_end))) {
        afsk_set_error("afsk_rx_plan_reset: bad argument");
        return AFSK_E_ARG;
    }
    AfskDeviceGuard guard(P->device);
    if (!guard.ok) { afsk_set_error("cannot select device %d", P->device); return AFSK_E_CUDA; }
    std::vector<int64_t> len;
    if (!h_len) {                                        // CSR offsets (B + 1)
        len.resize((size_t)B);
        for (int c = 0; c < B; c++) len[c] = h_start[c + 1] - h_start[c];
        h_len = len.data();
    }
    for (auto &ev : P->timing_events) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    P->timing_events.clear();
    P->timed_launches = 0;
    const int rc = plan_build(P, B, h_start, h_len, h_baud, h_amp_end);
    if (rc != AFSK_OK) { P->B = 0; P->groups.clear(); }  // unusable until the next successful reset
    return rc;
}

int afsk_rx_plan_destroy(AfskRxPlan *P)
{
    if (!P) return AFSK_OK;
    AfskDeviceGuard guard(P->device);
    for (auto &ev : P->timing_events) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    for (cudaStream_t gs : P->gstreams) cudaStreamDestroy(gs);
    for (cudaEvent_t ge : P->gevents) cudaEventDestroy(ge);
    cudaFree(P->arena);
    delete P;
    return AFSK_OK;
}

int afsk_rx_plan_set_option(AfskRxPlan *P, int option, int value)
{
    if (!P) return AFSK_E_ARG;
    switch (option) {
    case AFSK_OPT_FRAME_KERNEL:
        if (value < 0 || value > 4) { afsk_set_error("AFSK_OPT_FRAME_KERNEL: 0..4"); return AFSK_E_ARG; }
        P->frame_kernel = value;
        return AFSK_OK;
    case AFSK_OPT_L2_HINT:
        P->l2_hint = value < 0 ? -1 : (value ? 1 : 0);
        return AFSK_OK;
    case AFSK_OPT_GROUP_STREAMS:
        P->group_streams = value ? 1 : 0;
        return AFSK_OK;
    case AFSK_OPT_CLOCK_KERNEL:
        if (value < 0 || value > 2) { afsk_set_error("AFSK_OPT_CLOCK_KERNEL: 0, 1 or 2"); return AFSK_E_ARG; }
        P->clock_kernel = value;
        return AFSK_OK;
    case AFSK_OPT_FUSED:
        if (value > 2) { afsk_set_error("AFSK_OPT_FUSED: -1..2"); return AFSK_E_ARG; }
        P->fused = value < 0 ? -1 : value;
        return AFSK_OK;
    default:
        afsk_set_error("afsk_rx_plan_set_option: unknown option %d", option);
        return AFSK_E_ARG;
    }
}

int afsk_rx_plan_out_offsets(const AfskRxPlan *P, const int64_t **h_out_off)
{
    if (!P || !h_out_off) return AFSK_E_ARG;
    *h_out_off = P->out_off.data();
    return AFSK_OK;
}

// which schedule a decode of this plan uses (see "auxiliary warps"): 0 three kernels, 1 clocks recovered by the
// demodulator's auxiliary warps, 2 clocks and framing
static int plan_fused_level(const AfskRxPlan *P)
{
    if (!P->can_fuse || P->fused == 0) return 0;
    int level = P->fused;
    if (level < 0) {
        // automatic = three kernels.  Measured on B200, same box, alternating runs (profiles/r2_tuning_log.md):
        //   level 1 (fused clocks): c2 (602 K-frame captures) 0.768 ms against 0.768 — the 24 us of k_clock come back as
        //   a later start of the stream (the first tiles wait ~10 us for the first round of clock jobs) and as issue
        //   slots taken from the consumers; c3 (143 K-frame captures) 1.07 ms against 0.82: 55 clock jobs of ~8 us per
        //   CTA, 3,500 warp instructions each, in a kernel that is already short of issue slots.
        //   level 2 (fused framing too): c2 0.769 against 0.737, c3 1.05 against 0.81 — the consumer warps' reports cost
        //   two GPU-scope fences per 32 tiles, more than k_frame_warp takes on an idle GPU.
        level = 0;
    }
    if (level >= 2 && (P->max_windows > kFrameWarpMaxWindows || P->frame_kernel > 1)) level = 1;
    return level;
}
static bool plan_fused(const AfskRxPlan *P) { return plan_fused_level(P) >= 1; }
static bool plan_fused_frame(const AfskRxPlan *P) { return plan_fused_level(P) >= 2; }

// clock recovery launches of the three-kernel schedule (same selection as afsk_rx_decode)
static bool clock_q_group(const Group &g) { return !g.caps.empty() && g.bf % 4 == 0 && g.bf >= 8 && g.bf <= 24; }
static int plan_clock_launches(const AfskRxPlan *P)
{
    if (P->clock_kernel != 0) return 1;
    int n = 0;
    int64_t qcaps = 0;
    for (const Group &g : P->groups)
        if (clock_q_group(g)) { n++; qcaps += (int64_t)g.caps.size(); }
    return n + (qcaps < P->B ? 1 : 0);
}

int afsk_rx_plan_launches(const AfskRxPlan *P, int *launches)
{
    if (!P || !launches) return AFSK_E_ARG;
    if (P->B == 0) *launches = 0;
    else if (plan_fused(P)) *launches = (int)P->groups.size() + (P->n_preset > 0 ? 1 : 0) + (plan_fused_frame(P) ? 0 : 1);
    else *launches = plan_clock_launches(P) + 1 + (int)P->groups.size();
    return AFSK_OK;
}

int afsk_rx_plan_set_timing(AfskRxPlan *P, int enable)
{
    if (!P) return AFSK_E_ARG;
    P->timing = enable != 0;
    return AFSK_OK;
}

int afsk_rx_plan_demod_time(AfskRxPlan *P, float *ms_total, int *launches)
{
    if (!P || !ms_total || !launches) return AFSK_E_ARG;
    AfskDeviceGuard guard(P->device);
    float total = 0.f;
    int n = 0;
    for (auto &ev : P->timing_events) {
        float ms = 0.f;
        if (cudaEventSynchronize(ev.second) == cudaSuccess && cudaEventElapsedTime(&ms, ev.first, ev.second) == cudaSuccess) {
            total += ms;
            n++;
        }
        cudaEventDestroy(ev.first);
        cudaEventDestroy(ev.second);
    }
    P->timing_events.clear();
    *ms_total = total;
    *launches = P->timed_launches ? P->timed_launches : n;     // overlapped groups are timed as one span per decode
    P->timed_launches = 0;
    return AFSK_OK;
}

int afsk_rx_plan_planes(const AfskRxPlan *P, int capture, const uint32_t **d_planes, int64_t *max_windows)
{
    if (!P || capture < 0 || capture >= P->B) return AFSK_E_ARG;
    const CapDesc &d = P->caps[capture];
    if (d_planes) *d_planes = reinterpret_cast<const uint32_t *>(P->d_planes + d.plane_base);
    if (max_windows) *max_windows = d.status0 == 0 ? (d.n - d.bf + d.bf - 1) / d.bf : 0;
    return AFSK_OK;
}

// The framing launch of B captures (planes at caps[c].plane_base, clocks in clock[]): automatic by capture length
// (fk = 0), or forced (AFSK_OPT_FRAME_KERNEL) where the forced variant can represent the batch (k_frame_warp:
// <= 2^18 windows per capture; int indices: < 2^30)
static void launch_frame(int fk, int B, const CapDesc *caps, const int32_t *clock, const uint2 *planes, uint8_t *d_out,
                         AfskRxResult *d_res, int64_t max_windows, int64_t sum_windows, int64_t gpu_caps, cudaStream_t st)
{
    if (fk == 1 && max_windows > kFrameWarpMaxWindows) fk = 0;
    if ((fk == 2 || fk == 3) && max_windows >= ((int64_t)1 << 30)) fk = 0;
    if (fk == 0) {
        if (max_windows <= kFrameWarpMaxWindows) fk = 1;
        else if (max_windows >= ((int64_t)1 << 30)) fk = 4;
        else if (sum_windows > 65536 * std::max<int64_t>(gpu_caps, 1)) fk = 3;   // long captures on average
        else fk = 2;
    }
    if (fk == 1)
        k_frame_warp<<<(B + kFrameWarpCaps - 1) / kFrameWarpCaps, 32 * kFrameWarpCaps, 0, st>>>(caps, clock, planes, d_out, d_res, B);
    else if (fk == 4)
        k_frame<512, 8, long long><<<B, 512, 0, st>>>(caps, clock, planes, d_out, d_res);
    else if (fk == 3)
        k_frame<512, 8, int><<<B, 512, 0, st>>>(caps, clock, planes, d_out, d_res);
    else
        k_frame<128, 4, int><<<B, 128, 0, st>>>(caps, clock, planes, d_out, d_res);
}

int afsk_rx_decode(AfskRxPlan *P, const int16_t *d_samples, uint8_t *d_out, AfskRxResult *d_res, void *stream)
{
    if (!P || (P->B > 0 && (!d_samples || !d_out || !d_res))) { afsk_set_error("afsk_rx_decode: null argument"); return AFSK_E_ARG; }
    if ((reinterpret_cast<uintptr_t>(d_samples) & 15) != 0) { afsk_set_error("afsk_rx_decode: d_samples must be 16-byte aligned"); return AFSK_E_ARG; }
    if ((reinterpret_cast<uintptr_t>(d_out) & 3) != 0) { afsk_set_error("afsk_rx_decode: d_out must be 4-byte aligned"); return AFSK_E_ARG; }
    if (P->B == 0) return AFSK_OK;
    AfskDeviceGuard guard(P->device);
    if (!guard.ok) { afsk_set_error("cannot select device %d", P->device); return AFSK_E_CUDA; }
    cudaStream_t st = (cudaStream_t)stream;
    const bool fused = plan_fused(P), fused_frame = plan_fused_frame(P);
    if (fused) {
        P->epoch++;
        if (P->epoch == 0) P->epoch = 1;                 // tag 0 is what a fresh arena holds
        if (P->n_preset > 0) k_preset<<<(P->B + 255) / 256, 256, 0, st>>>(P->d_caps, P->d_clock, d_res, P->B);
    } else if (P->clock_kernel == 2 && P->can_clock2) {
        k_clock2<<<P->B, 128, 0, st>>>(d_samples, P->d_caps, P->d_clock, d_res);
    } else {
        // automatic: the short-bit groups through k_clock_q (registers only), everything else through k_clock, which
        // leaves the captures of those groups alone (and is not launched at all when they are the whole batch)
        uint32_t qmask = 0;
        int64_t qcaps = 0;
        if (P->clock_kernel == 0) {
            for (const Group &g : P->groups) {
                if (!clock_q_group(g)) continue;
                const int ng = (int)g.caps.size();
                switch (g.bf) {
                case 8: k_clock_q<2><<<ng, kClockThreads, 0, st>>>(d_samples, P->d_caps, g.d_caps, P->d_clock); break;
                case 12: k_clock_q<3><<<ng, kClockThreads, 0, st>>>(d_samples, P->d_caps, g.d_caps, P->d_clock); break;
                case 16: k_clock_q<4><<<ng, kClockThreads, 0, st>>>(d_samples, P->d_caps, g.d_caps, P->d_clock); break;
                case 20: k_clock_q<5><<<ng, kClockThreads, 0, st>>>(d_samples, P->d_caps, g.d_caps, P->d_clock); break;
                default: k_clock_q<6><<<ng, kClockThreads, 0, st>>>(d_samples, P->d_caps, g.d_caps, P->d_clock); break;
                }
                qmask |= 1u << (g.bf >> 2);
                qcaps += ng;
            }
        }
        if (qcaps < P->B) k_clock<<<P->B, kClockThreads, 0, st>>>(d_samples, P->d_caps, P->d_clock, d_res, qmask);
    }
    const int ngroups = (int)P->groups.size();
    const bool multi = P->group_streams != 0 && ngroups > 1;
    if (multi) {
        while ((int)P->gstreams.size() < ngroups - 1) {
            cudaStream_t gs;
            AFSK_CUDA(cudaStreamCreateWithFlags(&gs, cudaStreamNonBlocking));
            P->gstreams.push_back(gs);
        }
        while ((int)P->gevents.size() < ngroups) {
            cudaEvent_t ge;
            AFSK_CUDA(cudaEventCreateWithFlags(&ge, cudaEventDisableTiming));
            P->gevents.push_back(ge);
        }
    }
    cudaEvent_t span0 = nullptr, span1 = nullptr;      // timing of the whole demodulation when the groups overlap
    if (multi && P->timing && cudaEventCreate(&span0) == cudaSuccess && cudaEventCreate(&span1) == cudaSuccess)
        cudaEventRecord(span0, st);
    if (multi) AFSK_CUDA(cudaEventRecord(P->gevents[0], st));             // the clocks (and preset results) are in place
    for (int gi = 0; gi < ngroups; gi++) {
        const Group &g = P->groups[gi];
        cudaStream_t gs = (multi && gi > 0) ? P->gstreams[gi - 1] : st;
        if (multi && gi > 0) AFSK_CUDA(cudaStreamWaitEvent(gs, P->gevents[0], 0));
        DemodParams p;
        p.samples = d_samples; p.caps = P->d_caps; p.clock = P->d_clock;
        p.gcaps = g.d_caps; p.gtile_first = g.d_tile_first; p.tile_gpos = g.d_tile_gpos;
        p.planes = P->d_planes;
        p.ng = (int)g.caps.size(); p.total_items = g.tile_first.back();
        p.bf = g.bf; p.tpw_log2 = g.tpw_log2; p.seg = g.seg; p.nv = g.nv; p.nt = g.nt; p.merge = g.merge; p.wt = g.wt; p.nsub = g.nsub;
        // rotated vector order: 375 baud 4357 -> 4800 GB/s, 750 baud 4730 -> 4855; at 1500 baud (one thread per window) it loses
        // the amplitude-only treatment of the merged vector and with it 6 % (5690 -> 5340): off there
        p.rot = (P->rot && g.tpw_log2 >= 1) ? 1 : 0;
        p.stage_bytes = g.stage_bytes; p.stages = g.stages;
        // L2 evict-first on the bulk copies (the samples are read once).  Same-box A/B: k_demod +2-6 %
        // (c2 0.768 -> 0.745 ms, 600 baud 0.819 -> 0.770), k_demod_shift +1-2.5 %, the short-window kernel 0 to -10 %
        // depending on the box, so the short-window kernel keeps the default policy.  AFSK_L2_HINT=0/1 (environment, read at
        // plan creation) or AFSK_OPT_L2_HINT force it.
        p.l2_hint = P->l2_hint >= 0 ? P->l2_hint : (g.small_wpt ? 0 : 1);
        // producer warps of the padded layout, 16-vector segments (one CTA per SM), two boxes: 750 baud 5267 / 5841-5969 / 6118-6232 /
        // 5503 GB/s with 2 / 3 / 4 / 5 warps, 1500 baud 5757 / 5758-6120 / 6042-6055 / 5006, 375 baud - / 6026-6328 / 6339 / 5846-6054
        p.pad_warps = P->pad_warps > 0 ? P->pad_warps : 4;
        p.fused = fused ? 1 : 0; p.fused_frame = fused_frame ? 1 : 0;
        p.epoch = P->epoch; p.aux_off = g.aux_off; p.clk_magic = g.clk_magic; p.clk_shift = g.clk_shift;
        p.cready = P->d_cready; p.clock_out = P->d_clock; p.tiles_done = g.d_tiles_done; p.ctrl = g.d_ctrl;
        p.out = d_out; p.res = d_res;
        const int grid = fused ? g.grid_fused : g.grid;
        const int block = g.pad ? kFusedThreads4 : (!fused ? kDemodThreads : ((g.small_wpt || g.shift_wpt) ? kFusedThreads4 : kFusedThreads2));
        const size_t smem = fused ? g.smem_fused : g.smem;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (!multi && P->timing && cudaEventCreate(&e0) == cudaSuccess && cudaEventCreate(&e1) == cudaSuccess)
            cudaEventRecord(e0, gs);
        if (g.small_wpt && g.bf == 8) k_demod_lane<1, 8, 8><<<grid, block, smem, gs>>>(p);
        else if (g.small_wpt && g.bf == 16) k_demod_lane<2, 4, 8><<<grid, block, smem, gs>>>(p);
        else if (g.small_wpt && g.bf == 24) k_demod_lane<3, 2, 8><<<grid, block, smem, gs>>>(p);
#define X(BF, W) \
        else if (g.pad && g.shift_wpt == (W) && g.bf == (BF)) k_demod_shift<BF, W, true><<<grid, block, smem, gs>>>(p);
        AFSK_PAD_VARIANTS(X)
#undef X
#define X(BF, W) \
        else if (!g.pad && g.shift_wpt == (W) && g.bf == (BF)) k_demod_shift<BF, W><<<grid, block, smem, gs>>>(p);
        AFSK_SHIFT_VARIANTS(X)
#undef X
        else launch_demod(g.merge, g.nt, grid, block, smem, gs, p);
        if (e0 && e1) {
            cudaEventRecord(e1, gs);
            P->timing_events.emplace_back(e0, e1);
        }
        if (P->timing) P->timed_launches++;
        if (multi && gi > 0) {
            AFSK_CUDA(cudaEventRecord(P->gevents[gi], gs));
            AFSK_CUDA(cudaStreamWaitEvent(st, P->gevents[gi], 0));         // join: framing needs every group's planes
        }
    }
    if (span0 && span1) {
        cudaEventRecord(span1, st);
        P->timing_events.emplace_back(span0, span1);
    }
    if (fused_frame) {
        AFSK_CUDA(cudaGetLastError());
        return AFSK_OK;
    }
    launch_frame(P->frame_kernel, P->B, P->d_caps, P->d_clock, P->d_planes, d_out, d_res, P->max_windows, P->sum_windows, P->gpu_caps, st);
    AFSK_CUDA(cudaGetLastError());
    return AFSK_OK;
}

// afsk_rx_decode_host keeps one plan and one set of grow-only device / pinned buffers per device between
// calls (a drop-in Receiver.load calls it once per file): after the first call a decode costs the two
// copies and three launches, no allocation.  Calls on the same device are serialised by the context's mutex.
namespace {
struct HostCtx {
    std::mutex m;
    AfskRxPlan *plan = nullptr;
    int16_t *d_samples = nullptr; size_t samples_cap = 0;
    uint8_t *d_out = nullptr; size_t out_cap = 0;
    AfskRxResult *d_res = nullptr; size_t res_cap = 0;
    uint8_t *h_stage = nullptr; size_t stage_cap = 0;      // pinned: results, then the payload blob
};
HostCtx g_host_ctx[64];

}  // namespace

int afsk_rx_decode_host(int device, const int16_t *h_samples, const int64_t *h_offsets, int B, const int32_t *h_baud,
                        const int32_t *h_amp_end, uint8_t *h_out, const int64_t *h_out_off, AfskRxResult *h_res)
{
    if (B < 0 || (B > 0 && (!h_samples || !h_offsets || !h_out || !h_out_off || !h_res))) return AFSK_E_ARG;
    if (B == 0) return AFSK_OK;
    if (device < 0 || device >= 64) { afsk_set_error("afsk_rx_decode_host: device %d out of range", device); return AFSK_E_ARG; }
    HostCtx &X = g_host_ctx[device];
    std::lock_guard<std::mutex> lock(X.m);
    int rc;
    if (!X.plan) rc = afsk_rx_plan_create(device, B, h_offsets, h_baud, h_amp_end, &X.plan);
    else rc = afsk_rx_plan_reset(X.plan, B, h_offsets, nullptr, h_baud, h_amp_end);
    if (rc) return rc;
    AfskRxPlan *P = X.plan;
    AfskDeviceGuard guard(device);
    const int64_t total = h_offsets[B], base = h_offsets[0] & ~(int64_t)7;
    const size_t sample_bytes = (size_t)(((total - base) * 2 + 15) & ~(int64_t)15) + 16;
    const size_t out_bytes = (size_t)P->out_off[B], res_bytes = sizeof(AfskRxResult) * (size_t)B;
    cudaError_t e = grow_device((void **)&X.d_samples, &X.samples_cap, sample_bytes);
    if (e == cudaSuccess) e = grow_device((void **)&X.d_out, &X.out_cap, out_bytes);
    if (e == cudaSuccess) e = grow_device((void **)&X.d_res, &X.res_cap, res_bytes);
    if (e == cudaSuccess && res_bytes + out_bytes > X.stage_cap) {
        if (X.h_stage) cudaFreeHost(X.h_stage);
        X.h_stage = nullptr; X.stage_cap = 0;
        const size_t want = (res_bytes + out_bytes) * 5 / 4 + 4096;
        e = cudaMallocHost((void **)&X.h_stage, want);
        if (e == cudaSuccess) X.stage_cap = want;
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(X.d_samples, h_samples + base, (size_t)(total - base) * 2, cudaMemcpyHostToDevice, 0);
    if (e == cudaSuccess) {
        // the plan indexes samples from global sample 0: pass the shifted base pointer
        rc = afsk_rx_decode(P, X.d_samples - base, X.d_out, X.d_res, nullptr);
        if (rc == AFSK_OK) {
            AfskRxResult *sr = reinterpret_cast<AfskRxResult *>(X.h_stage);
            uint8_t *sb = X.h_stage + res_bytes;
            e = cudaMemcpyAsync(sr, X.d_res, res_bytes, cudaMemcpyDeviceToHost, 0);
            if (e == cudaSuccess) e = cudaMemcpyAsync(sb, X.d_out, out_bytes, cudaMemcpyDeviceToHost, 0);
            if (e == cudaSuccess) e = cudaStreamSynchronize(0);
            if (e == cudaSuccess) {
                memcpy(h_res, sr, res_bytes);
                // compact copy-back: only the decoded bytes of each capture
                for (int c = 0; c < B; c++) {
                    int64_t nb = sr[c].nbytes, cap = h_out_off[c + 1] - h_out_off[c];
                    if (nb > cap) { rc = AFSK_E_ARG; afsk_set_error("output capacity too small for capture %d", c); break; }
                    if (nb > 0) memcpy(h_out + h_out_off[c], sb + P->out_off[c], (size_t)nb);
                }
            }
        }
    }
    if (e != cudaSuccess) { afsk_set_error("afsk_rx_decode_host: %s", cudaGetErrorString(e)); return AFSK_E_CUDA; }
    return rc;
}

#ifdef AFSK_DBG_TRACE
int afsk_dbg_trace_read(unsigned long long *h_out, int max_records, int reset)
{
    unsigned int n = 0;
    cudaMemcpyFromSymbol(&n, g_trace_n, sizeof(n));
    if (n > (1u << 12)) n = 1u << 12;
    if ((int)n > max_records) n = (unsigned)max_records;
    if (n) cudaMemcpyFromSymbol(h_out, g_trace, sizeof(unsigned long long) * 10 * n);
    if (reset) { unsigned int z = 0; cudaMemcpyToSymbol(g_trace_n, &z, sizeof(z)); }
    return (int)n;
}
#endif

/* releases what afsk_rx_decode_host keeps per device between calls */
int afsk_rx_host_release(int device)
{
    if (device < 0 || device >= 64) return AFSK_E_ARG;
    HostCtx &X = g_host_ctx[device];
    std::lock_guard<std::mutex> lock(X.m);
    AfskDeviceGuard guard(device);
    if (X.plan) afsk_rx_plan_destroy(X.plan);
    X.plan = nullptr;
    cudaFree(X.d_samples); cudaFree(X.d_out); cudaFree(X.d_res);
    if (X.h_stage) cudaFreeHost(X.h_stage);
    X.d_samples = nullptr; X.d_out = nullptr; X.d_res = nullptr; X.h_stage = nullptr;
    X.samples_cap = X.out_cap = X.res_cap = X.stage_cap = 0;
    return AFSK_OK;
}

int afsk_rx_gate(int device, const int16_t *d_samples, const int64_t *h_offsets, int S, int amp_start, int amp_end,
                 int64_t timeout_frames, int64_t *d_range, void *stream)
{
    if (S < 0 || (S > 0 && (!d_samples || !h_offsets || !d_range))) { afsk_set_error("afsk_rx_gate: bad argument"); return AFSK_E_ARG; }
    return gate_run(device, d_samples, h_offsets, S, amp_start, amp_end, timeout_frames, -1, d_range, nullptr, stream);
}

int afsk_rx_gate_multi(int device, const int16_t *d_samples, const int64_t *h_offsets, int S, int amp_start, int amp_end,
                       int64_t timeout_frames, int max_calls, int64_t *d_ranges, int32_t *d_counts, void *stream)
{
    if (S < 0 || max_calls < 0 || (S > 0 && (!d_samples || !h_offsets || !d_ranges || !d_counts))) {
        afsk_set_error("afsk_rx_gate_multi: bad argument");
        return AFSK_E_ARG;
    }
    return gate_run(device, d_samples, h_offsets, S, amp_start, amp_end, timeout_frames, max_calls, d_ranges, d_counts, stream);
}

// ---------------------------------------------------------------- streaming receiver ----
// S channels, each one Receiver calling receive(timeout) again and again on its own open input stream,
// fed piece by piece.  Every channel keeps its samples from its pending recording's first chunk (or,
// with none, from its partial chunk) on in a slot of a device arena.  A push appends the pieces
// (k_stream_copy), measures the chunks they completed (k_gate_amp), resumes every channel's walk
// (k_gate_multi) and decodes the recordings that became final in place, through one plan re-targeted
// with afsk_rx_plan_reset.
//
// Retention moves only the channel whose piece does not fit behind its slot.  Its retained samples go back
// to the start of its slot when they fill at most half of it, else into a new slot of twice its need (plus
// two chunks) at the top of the arena.  Only when the top has no room for those does every channel move,
// into the other arena: slots of twice their need, and half as much again free above them.  A move costs
// at most the frames its channel pushed since the slot was assigned, and a compaction moves at most what
// the channels pushed while the free space filled, so every pushed frame causes O(1) moved frames
// (afsk_rx_streams_counters reports them), and one long recording widens only its own slot.
//
// Retention mode AFSK_RETAIN_BITS demodulates open recordings as they arrive instead.  Once 4096 frames of a
// pending recording are in, its clock is recovered (k_clock_q / k_clock, as a plan chooses them) and stored;
// from then on every push decides the recording's complete 32-window plane words (k_stream_windows) into the
// channel's slot of a plane arena, which follows the same policy as the sample arena (a plane word counts as
// four samples).  The channel keeps its samples only from its first undecided window, or from its partial
// chunk if that is earlier.  When the recording becomes final, its remaining windows are decided from that tail
// and it is framed from its planes (k_frame_warp / k_frame).  A recording that ends before its clock is stored
// still has all its samples and is decoded through the plan.  Each window's bit and quiet flag depend on its
// own samples only, and the final length only decides how many windows count, so the results are the same.
//
// Retention mode AFSK_RETAIN_PAYLOAD also frames such a recording push by push (k_stream_frame) over its windows below
// K_safe = windows_of((g.pos - mark) * 2048, bf, clock), which every later end of the recording includes (it ends at a
// closing quiet chunk at or after g.pos, or a finish cuts it at its last full chunk), as far as they are decided.  The
// channel then keeps plane words only from the one its search or its next incomplete byte needs, and its decoded bytes
// in a payload slot (a third arena with the same policy, two bytes counting as one sample); once the first quiet window
// after the terminator is found the result is fixed, and it decides no more windows, keeps no planes and keeps samples
// only from its partial chunk.  When the recording becomes final, the same kernel frames the rest up to its K and
// writes the result as k_frame does.
namespace {
constexpr int64_t kSlotPad = 64;           // samples after the last slot (vector over-reads of the kernels)
int64_t arena_frames(size_t bytes) { return bytes ? (int64_t)(bytes / 2) - kSlotPad : 0; }

// an arena pair with one slot per channel, in samples (a plane word is four)
struct Slots {
    // per channel: first arena sample, capacity, stream position at the slot's start
    std::vector<int64_t> off, cap, base;
    int16_t *arena[2] = {nullptr, nullptr};
    size_t arena_cap[2] = {0, 0};
    int cur = 0;
    int64_t top = 0;                                              // arena samples below the free space
    int64_t n_moved = 0, n_compactions = 0;                       // since creation
};

void add_seg(CopySeg *seg, int64_t *tf, int &n, int64_t src, int64_t dst, int64_t len)
{
    if (len <= 0) return;
    const int64_t vecs = ((dst + len + 7) >> 3) - (dst >> 3);
    seg[n] = CopySeg{src, dst, len};
    tf[n + 1] = tf[n] + (vecs + kCopyTileVecs - 1) / kCopyTileVecs;
    n++;
}

// The retention step of one push (see above) for channels that have pushed[s], will have np[s] and keep from
// keep[s] on: assigns the slots and lists the moves of the retained spans [keep[s], pushed[s]).  A compaction
// allocates the other arena first; a failed allocation leaves A as it was.
cudaError_t slots_retain(Slots &A, int S, const int64_t *pushed, const int64_t *np, const int64_t *keep, int64_t *new_off,
                         int64_t *new_cap, CopySeg *seg, int64_t *tf, int &nmov, bool &compact)
{
    const int64_t C = AFSK_GATE_CHUNK;
    auto overflows = [&](int s) { return np[s] - A.base[s] > A.cap[s]; };
    auto rewinds = [&](int s) { return 2 * (np[s] - keep[s]) <= A.cap[s]; };
    auto fresh_cap = [&](int s) { return (2 * (np[s] - keep[s]) + 2 * C + 7) & ~(int64_t)7; };
    int64_t want = 0;
    bool any = false;
    for (int s = 0; s < S; s++)
        if (overflows(s)) {
            any = true;
            if (!rewinds(s)) want += fresh_cap(s);
        }
    compact = any && A.top + want > arena_frames(A.arena_cap[A.cur]);
    nmov = 0;
    tf[0] = 0;
    if (compact) {
        int64_t total = 0;
        for (int s = 0; s < S; s++) {
            new_off[s] = total;
            new_cap[s] = fresh_cap(s);
            total += new_cap[s];
        }
        const int nxt = A.cur ^ 1;
        const cudaError_t e = grow_device((void **)&A.arena[nxt], &A.arena_cap[nxt], (size_t)(total + total / 2 + kSlotPad) * 2);
        if (e != cudaSuccess) return e;
        for (int s = 0; s < S; s++) {
            add_seg(seg, tf, nmov, A.off[s] + keep[s] - A.base[s], new_off[s], pushed[s] - keep[s]);
            A.off[s] = new_off[s]; A.cap[s] = new_cap[s]; A.base[s] = keep[s];
        }
        A.top = total;
        A.n_compactions++;
    } else if (any) {
        // within the arena: sources are the retained spans, destinations the slot starts (below the span: a
        // rewind happens only when the span fills at most half the slot) or fresh space above the top
        for (int s = 0; s < S; s++) {
            if (!overflows(s)) continue;
            const int64_t src = A.off[s] + keep[s] - A.base[s];
            if (!rewinds(s)) {
                A.off[s] = A.top;
                A.cap[s] = fresh_cap(s);
                A.top += A.cap[s];
            }
            add_seg(seg, tf, nmov, src, A.off[s], pushed[s] - keep[s]);
            A.base[s] = keep[s];
        }
    }
    for (int i = 0; i < nmov; i++) A.n_moved += seg[i].len;
    return cudaSuccess;
}

// the moves slots_retain listed (descriptors already on the device), then the compacted arena becomes current
void slots_move(Slots &A, bool compact, int nmov, const uint8_t *d_seg, const uint8_t *d_tf, int64_t tiles, cudaStream_t st,
                int64_t &launches)
{
    if (nmov > 0) {
        k_stream_copy<<<(unsigned)tiles, kCopyThreads, 0, st>>>(A.arena[A.cur], A.arena[compact ? A.cur ^ 1 : A.cur],
                                                                reinterpret_cast<const CopySeg *>(d_seg),
                                                                reinterpret_cast<const int64_t *>(d_tf), nmov);
        launches++;
    }
    if (compact) A.cur ^= 1;
}

// K = #{k >= 0 : clk + k bf < n - bf}, as num_windows
int64_t windows_of(int64_t n, int bf, int64_t clk)
{
    const int64_t span = n - bf - clk;
    return span <= 0 ? 0 : (span + bf - 1) / bf;
}

// what bits mode does with a channel's recordings at this baud: > 0, the bit length: demodulated as they arrive;
// 0: decided from length and baud alone (k_preset's statuses: no sample is needed); -1: kept whole
int bits_bf(int baud)
{
    int bf, ml, sl;
    if (!afsk_tone_geometry(baud, &bf, &ml, &sl) || AFSK_SYNC_FRAMES - 2 * bf <= 0 || ml != bf || sl != bf) return 0;
    return (bf % 4 == 0 && bf <= kWinMaxBf) ? bf : -1;
}

int32_t clamp_thr(int32_t amp_end) { return std::min<int32_t>(std::max<int32_t>(amp_end, 0), 65537); }
}  // namespace

struct AfskRxStreams {
    int device = 0, S = 0;
    // per channel: the receiver's baud, and its gate settings (host copy of d_params)
    std::vector<int32_t> baud;
    std::vector<GateParams> params;
    GateParams *d_params = nullptr;
    // per channel (host): frames pushed, first retained frame, start of the pending recording (-1: none), calls
    // finished; the sample slots
    std::vector<int64_t> pushed, keep, pending, calls;
    Slots smp;
    std::vector<int64_t> np, new_off, new_cap, chunk_first;       // scratch of one push
    bool failed = false;                                          // an error after this push's state was committed
    bool used = false;                                            // a push or finish has run (the retention mode is fixed)
    int retain = AFSK_RETAIN_SAMPLES;
    int64_t n_launches = 0;                                       // since creation
    int16_t *d_stage = nullptr; size_t stage_cap = 0;             // host input
    // descriptors of one push, built in pinned memory and sent with one copy
    uint8_t *d_desc = nullptr, *h_desc = nullptr;
    // (the finish flags come last: a push copies the block up to o_fin only)
    size_t desc_bytes = 0, o_seg_app = 0, o_tf_app = 0, o_seg_mov = 0, o_tf_mov = 0, o_first = 0, o_amp_off = 0, o_out_first = 0,
           o_fin = 0;
    GateState *d_state = nullptr, *h_state = nullptr;
    int32_t *d_counts = nullptr, *h_counts = nullptr;
    int32_t *d_amp = nullptr; size_t amp_cap = 0;
    int64_t *d_ranges = nullptr, *h_ranges = nullptr; size_t ranges_cap = 0, h_ranges_cap = 0;
    AfskRxPlan *plan = nullptr;
    uint8_t *d_out = nullptr; size_t out_cap = 0;
    AfskRxResult *d_res = nullptr; size_t res_cap = 0;
    uint8_t *h_dec = nullptr; size_t h_dec_cap = 0;               // pinned: results, then payloads
    std::vector<int64_t> rec_start, rec_len;
    std::vector<int32_t> rec_baud, rec_amp_end;
    // bits mode, per channel: the pending recording's clock (-1: not stored), its windows decided, and the channel's
    // plane stream (in samples, four per word): where the recording's window 0 lies, the end used, the first kept
    std::vector<int64_t> pclock, pdecided, pw_rec, pw_pushed, pw_keep;
    Slots pln;
    // bits mode: descriptors (clock captures, their k_clock_q lists, plane moves, window jobs, frame captures and
    // clocks), clocks read back, framing output
    uint8_t *d_bdesc = nullptr, *h_bdesc = nullptr;
    size_t bdesc_bytes = 0, o_ccap = 0, o_cq = 0, o_clk = 0, o_seg_pmov = 0, o_tf_pmov = 0, o_win = 0, o_tf_win = 0, o_fcap = 0,
           o_fclk = 0;
    uint8_t *d_fout = nullptr; size_t fout_cap = 0;
    AfskRxResult *d_fres = nullptr; size_t fres_cap = 0;
    uint8_t *h_fdec = nullptr; size_t h_fdec_cap = 0;
    // payload mode, per channel: the framing state of the pending recording (h_fst: as the last push left it), and the
    // channel's payload stream (in samples, two bytes each): where the recording's byte 0 lies, the end used, the first
    // kept; descriptors (payload moves, frame jobs) in the bits-mode block
    FrameState *d_fst = nullptr, *h_fst = nullptr;
    std::vector<int64_t> py_rec, py_pushed, py_keep;
    Slots pay;
    size_t o_seg_ymov = 0, o_tf_ymov = 0, o_fjob = 0;
    // what the last push / finish returned
    std::vector<AfskRxStreamEvent> ev;
    std::vector<AfskRxResult> res;
    std::vector<uint8_t> payload;
    std::vector<int64_t> payload_off;
};

static int streams_fail(cudaError_t e)
{
    afsk_set_error("afsk_rx_streams: %s", cudaGetErrorString(e));
    return AFSK_E_CUDA;
}

// decodes H->rec_* (recordings as ranges of the sample arena) through the plan; *rr / *oo: results and payload offsets
// in H->h_dec, whose payloads start at *res_bytes.  Synchronizes st.
static int streams_decode_plan(AfskRxStreams *H, const int16_t *x, cudaStream_t st, const AfskRxResult **rr, const int64_t **oo,
                               size_t *res_bytes)
{
    const int nrec = (int)H->rec_start.size();
    int rc = H->plan ? afsk_rx_plan_reset(H->plan, nrec, H->rec_start.data(), H->rec_len.data(), H->rec_baud.data(), H->rec_amp_end.data())
                     : afsk_rx_plan_create_ranges(H->device, nrec, H->rec_start.data(), H->rec_len.data(), H->rec_baud.data(),
                                                  H->rec_amp_end.data(), &H->plan);
    if (rc != AFSK_OK) return rc;
    *oo = H->plan->out_off.data();
    const size_t rb = sizeof(AfskRxResult) * (size_t)nrec, out_bytes = (size_t)(*oo)[nrec];
    cudaError_t e = grow_device((void **)&H->d_out, &H->out_cap, out_bytes);
    if (e == cudaSuccess) e = grow_device((void **)&H->d_res, &H->res_cap, rb);
    if (e == cudaSuccess) e = grow_pinned((void **)&H->h_dec, &H->h_dec_cap, rb + out_bytes);
    if (e != cudaSuccess) return streams_fail(e);
    rc = afsk_rx_decode(H->plan, x, H->d_out, H->d_res, st);
    if (rc != AFSK_OK) return rc;
    int nl = 0;
    afsk_rx_plan_launches(H->plan, &nl);
    H->n_launches += nl;
    AFSK_CUDA(cudaMemcpyAsync(H->h_dec, H->d_res, rb, cudaMemcpyDeviceToHost, st));
    AFSK_CUDA(cudaMemcpyAsync(H->h_dec + rb, H->d_out, out_bytes, cudaMemcpyDeviceToHost, st));
    AFSK_CUDA(cudaStreamSynchronize(st));
    *rr = reinterpret_cast<const AfskRxResult *>(H->h_dec);
    *res_bytes = rb;
    return AFSK_OK;
}

static int streams_bits(AfskRxStreams *H, cudaStream_t st, const int64_t *out_first);

// one push (fin == NULL) or the end of the streams s with fin[s] != 0 (no samples); then, when new_baud is
// given, every channel's settings become new_baud[s] / new_params[s] for its next stream.  A push is planar
// (inter < 0: channel s's piece is samples[off[s] .. off[s + 1]), int16) or interleaved (inter frames of every
// channel, samples[f * pitch + s] = frame f of channel s in the AFSK_SAMPLE_* format; off unused)
static int streams_run(AfskRxStreams *H, const void *samples, int on_device, const int64_t *off, int64_t inter, int format,
                       int64_t pitch, cudaStream_t st, const uint8_t *fin, const int32_t *new_baud, const GateParams *new_params,
                       int64_t *n_events)
{
    const int S = H->S;
    const bool finish = fin != nullptr, interleaved = inter >= 0;
    const int64_t C = AFSK_GATE_CHUNK;
    auto piece = [&](int s) -> int64_t { return finish ? 0 : interleaved ? inter : off[s + 1] - off[s]; };
    int64_t nch = 0;                               // chunks completed by this push
    for (int s = 0; s < S; s++) {
        H->np[s] = H->pushed[s] + piece(s);
        nch += H->np[s] / C - H->pushed[s] / C;
    }
    // buffers first: a failed allocation leaves the channels as they were
    const int64_t in_samples = finish ? 0 : interleaved ? inter * S : off[S] - off[0];
    const int size = interleaved ? afsk_sample_size(format) : 2;
    cudaError_t e = cudaSuccess;
    if (!on_device && in_samples > 0) e = grow_device((void **)&H->d_stage, &H->stage_cap, (size_t)in_samples * size + 32);
    if (e == cudaSuccess) e = grow_device((void **)&H->d_amp, &H->amp_cap, sizeof(int32_t) * (size_t)nch);
    if (e == cudaSuccess) e = grow_device((void **)&H->d_ranges, &H->ranges_cap, sizeof(int64_t) * 3 * (size_t)(nch + S));
    if (e == cudaSuccess) e = grow_pinned((void **)&H->h_ranges, &H->h_ranges_cap, sizeof(int64_t) * 3 * (size_t)(nch + S));
    if (e != cudaSuccess) return streams_fail(e);
    uint8_t *hd = H->h_desc;
    CopySeg *seg_app = reinterpret_cast<CopySeg *>(hd + H->o_seg_app), *seg_mov = reinterpret_cast<CopySeg *>(hd + H->o_seg_mov);
    int64_t *tf_app = reinterpret_cast<int64_t *>(hd + H->o_tf_app), *tf_mov = reinterpret_cast<int64_t *>(hd + H->o_tf_mov);
    int64_t *first = reinterpret_cast<int64_t *>(hd + H->o_first), *amp_off = reinterpret_cast<int64_t *>(hd + H->o_amp_off);
    int64_t *out_first = reinterpret_cast<int64_t *>(hd + H->o_out_first);
    int nmov = 0, napp = 0;
    bool compact = false;
    e = slots_retain(H->smp, S, H->pushed.data(), H->np.data(), H->keep.data(), H->new_off.data(), H->new_cap.data(), seg_mov, tf_mov,
                     nmov, compact);
    if (e != cudaSuccess) return streams_fail(e);
    Slots &A = H->smp;
    tf_app[0] = 0;
    first[0] = 0;
    // interleaved device input is read from the 16-byte vector holding its first sample, e0 samples in; host input
    // is copied packed (pitch S) into the staging buffer
    const int e0 = interleaved && on_device ? (int)((reinterpret_cast<uintptr_t>(samples) & 15) / size) : 0;
    const int64_t kpitch = on_device ? pitch : S;                 // the pitch the kernel reads
    for (int s = 0; s < S; s++) {
        // (interleaved: src is the channel's column, which only a one-channel contiguous int16 push reads as a
        // k_stream_copy segment)
        const int64_t src = finish ? 0 : interleaved ? e0 + s : off[s] - (on_device ? 0 : off[0]);
        add_seg(seg_app, tf_app, napp, src, A.off[s] + H->pushed[s] - A.base[s], piece(s));
        const int64_t c_old = H->pushed[s] / C;
        first[s + 1] = first[s] + H->np[s] / C - c_old;
        amp_off[s] = A.off[s] + c_old * C - A.base[s];
        out_first[s] = first[s] + s;
    }
    if (finish) memcpy(hd + H->o_fin, fin, (size_t)S);
    AFSK_CUDA(cudaMemcpyAsync(H->d_desc, H->h_desc, finish ? H->desc_bytes : H->o_fin, cudaMemcpyHostToDevice, st));
    const uint8_t *dd = H->d_desc;
    slots_move(A, compact, nmov, dd + H->o_seg_mov, dd + H->o_tf_mov, tf_mov[nmov], st, H->n_launches);
    int16_t *x = A.arena[A.cur];
    if (napp > 0) {
        const void *src = on_device ? reinterpret_cast<const void *>(reinterpret_cast<uintptr_t>(samples) & ~(uintptr_t)15) : H->d_stage;
        if (!on_device && interleaved) {
            AFSK_CUDA(cudaMemcpy2DAsync(H->d_stage, (size_t)S * size, samples, (size_t)pitch * size, (size_t)S * size, (size_t)inter,
                                        cudaMemcpyHostToDevice, st));
        } else if (!on_device) {
            AFSK_CUDA(cudaMemcpyAsync(H->d_stage, static_cast<const int16_t *>(samples) + off[0], (size_t)in_samples * 2,
                                      cudaMemcpyHostToDevice, st));
        }
        const CopySeg *sg = reinterpret_cast<const CopySeg *>(dd + H->o_seg_app);
        if (interleaved && (S > 1 || format != AFSK_SAMPLE_S16 || kpitch != 1)) {
            const int cblocks = (S + kDiC - 1) / kDiC;
            const unsigned grid = (unsigned)(cblocks * ((inter + kDiF + kDiHalo - 1) / kDiF));
            if (format == AFSK_SAMPLE_S16 && kpitch == S && e0 == 0)
                k_stream_deinterleave<<<grid, kDiThreads, 0, st>>>(static_cast<const int16_t *>(src), x, sg, S, inter, cblocks);
            else if (format == AFSK_SAMPLE_S16)
                k_stream_frames<<<grid, kDiThreads, 0, st>>>(static_cast<const int16_t *>(src), x, sg, S, inter, kpitch, e0, cblocks);
            else if (format == AFSK_SAMPLE_S32)
                k_stream_frames<<<grid, kDiThreads, 0, st>>>(static_cast<const int32_t *>(src), x, sg, S, inter, kpitch, e0, cblocks);
            else
                k_stream_frames<<<grid, kDiThreads, 0, st>>>(static_cast<const float *>(src), x, sg, S, inter, kpitch, e0, cblocks);
        } else {
            k_stream_copy<<<(unsigned)tf_app[napp], kCopyThreads, 0, st>>>(static_cast<const int16_t *>(src), x, sg,
                                                                          reinterpret_cast<const int64_t *>(dd + H->o_tf_app), napp);
        }
        H->n_launches++;
    }
    const int64_t *d_first = reinterpret_cast<const int64_t *>(dd + H->o_first);
    if (nch > 0) {
        const int wpb = 8;
        k_gate_amp<<<(unsigned)((nch + wpb - 1) / wpb), wpb * 32, 0, st>>>(x, d_first, reinterpret_cast<const int64_t *>(dd + H->o_amp_off),
                                                                           S, nch, H->d_amp);
        H->n_launches++;
    }
    H->n_launches++;
    k_gate_multi<<<S, 32, 0, st>>>(H->d_amp, d_first, GateParams{}, H->d_params, 0x7FFFFFFF, H->d_state, 0,
                                   finish ? dd + H->o_fin : nullptr, reinterpret_cast<const int64_t *>(dd + H->o_out_first),
                                   H->d_ranges, H->d_counts);
    AFSK_CUDA(cudaGetLastError());
    AFSK_CUDA(cudaMemcpyAsync(H->h_counts, H->d_counts, sizeof(int32_t) * S, cudaMemcpyDeviceToHost, st));
    AFSK_CUDA(cudaMemcpyAsync(H->h_state, H->d_state, sizeof(GateState) * S, cudaMemcpyDeviceToHost, st));
    AFSK_CUDA(cudaMemcpyAsync(H->h_ranges, H->d_ranges, sizeof(int64_t) * 3 * (size_t)(nch + S), cudaMemcpyDeviceToHost, st));
    AFSK_CUDA(cudaStreamSynchronize(st));

    if (H->retain != AFSK_RETAIN_SAMPLES) {
        const int rc = streams_bits(H, st, out_first);
        if (rc != AFSK_OK) return rc;
    } else {
        // final calls, ordered by (channel, call); recordings as ranges of the arena
        H->ev.clear();
        H->rec_start.clear();
        H->rec_len.clear();
        H->rec_baud.clear();
        H->rec_amp_end.clear();
        for (int s = 0; s < S; s++) {
            const int64_t *r = H->h_ranges + 3 * out_first[s];
            for (int k = 0; k < H->h_counts[s]; k++) {
                AfskRxStreamEvent v;
                v.stream = s; v.recorded = (int32_t)r[3 * k]; v.call = H->calls[s] + k; v.start = r[3 * k + 1]; v.end = r[3 * k + 2];
                H->ev.push_back(v);
                if (v.recorded) {
                    H->rec_start.push_back(A.off[s] + v.start - A.base[s]);
                    H->rec_len.push_back(v.end - v.start);
                    H->rec_baud.push_back(H->baud[s]);
                    H->rec_amp_end.push_back(H->params[s].amp_end);
                }
            }
            const GateState &g = H->h_state[s];
            H->calls[s] = g.call;
            H->pushed[s] = H->np[s];
            H->pending[s] = g.phase == 2 ? g.mark * C : -1;
            H->keep[s] = g.phase == 2 ? g.mark * C : g.pos * C;
        }
        const int nev = (int)H->ev.size(), nrec = (int)H->rec_start.size();
        H->res.assign((size_t)nev, AfskRxResult{0, -1, -1, 0, 0});
        H->payload_off.assign((size_t)nev + 1, 0);
        H->payload.clear();
        if (nrec > 0) {
            const AfskRxResult *rr = nullptr;
            const int64_t *oo = nullptr;
            size_t res_bytes = 0;
            const int rc = streams_decode_plan(H, x, st, &rr, &oo, &res_bytes);
            if (rc != AFSK_OK) return rc;
            H->payload.assign(H->h_dec + res_bytes, H->h_dec + res_bytes + oo[nrec]);
            int k = 0;
            for (int i = 0; i < nev; i++) {
                H->payload_off[i] = oo[k];
                if (H->ev[i].recorded) H->res[i] = rr[k++];
            }
            H->payload_off[nev] = oo[nrec];
        }
    }
    if (finish)                                    // the next push is frame 0 of a new stream (k_gate_multi reset its state)
        for (int s = 0; s < S; s++)
            if (fin[s]) {
                H->pushed[s] = H->keep[s] = H->calls[s] = A.base[s] = 0;
                H->pending[s] = -1;
                if (H->retain != AFSK_RETAIN_SAMPLES) {
                    H->pclock[s] = -1;
                    H->pdecided[s] = H->pw_rec[s] = H->pw_pushed[s] = H->pw_keep[s] = H->pln.base[s] = 0;
                    H->py_rec[s] = H->py_pushed[s] = H->py_keep[s] = H->pay.base[s] = 0;
                }
            }
    if (new_baud) {
        AFSK_CUDA(cudaMemcpyAsync(H->d_params, new_params, sizeof(GateParams) * S, cudaMemcpyHostToDevice, st));
        AFSK_CUDA(cudaStreamSynchronize(st));
        H->baud.assign(new_baud, new_baud + S);
        H->params.assign(new_params, new_params + S);
    }
    *n_events = (int64_t)H->ev.size();
    return AFSK_OK;
}

// The rest of a bits- or payload-mode push, after the gate: the final calls (a recording that was pending with its
// clock stored is framed from its planes, any other through the plan), clocks of the pending recordings that now have
// 4096 frames, the plane slots, the windows decided, and the channels' new state.  In payload mode the recordings
// pending with a stored clock are also framed as far as the chunks the gate has walked (k_stream_frame, which frames
// the final ones too), and a recording whose first quiet window was found decides no more windows.
static int streams_bits(AfskRxStreams *H, cudaStream_t st, const int64_t *out_first)
{
    const int S = H->S;
    const int64_t C = AFSK_GATE_CHUNK;
    const bool pmode = H->retain == AFSK_RETAIN_PAYLOAD;
    Slots &A = H->smp, &Pl = H->pln, &Y = H->pay;
    const int16_t *x = A.arena[A.cur];
    uint8_t *hb = H->h_bdesc;
    const uint8_t *db = H->d_bdesc;
    CapDesc *ccap = reinterpret_cast<CapDesc *>(hb + H->o_ccap), *fcap = reinterpret_cast<CapDesc *>(hb + H->o_fcap);
    int32_t *cq = reinterpret_cast<int32_t *>(hb + H->o_cq), *fclk = reinterpret_cast<int32_t *>(hb + H->o_fclk);
    int32_t *h_clk = reinterpret_cast<int32_t *>(hb + H->o_clk);
    CopySeg *seg_pmov = reinterpret_cast<CopySeg *>(hb + H->o_seg_pmov);
    int64_t *tf_pmov = reinterpret_cast<int64_t *>(hb + H->o_tf_pmov), *tf_win = reinterpret_cast<int64_t *>(hb + H->o_tf_win);
    WinJob *win = reinterpret_cast<WinJob *>(hb + H->o_win);
    CopySeg *seg_ymov = reinterpret_cast<CopySeg *>(hb + H->o_seg_ymov);
    int64_t *tf_ymov = reinterpret_cast<int64_t *>(hb + H->o_tf_ymov);
    FrameJob *fjob = reinterpret_cast<FrameJob *>(hb + H->o_fjob);

    // final calls, ordered by (channel, call): src[i] >= 0 plan capture, <= -2 frame capture -2 - src[i], -1 none
    H->ev.clear();
    H->rec_start.clear();
    H->rec_len.clear();
    H->rec_baud.clear();
    H->rec_amp_end.clear();
    std::vector<int> src, fch(S, -1), fev;         // fch[s]: the channel's frame capture, fev[j]: its event
    int nf = 0;
    for (int s = 0; s < S; s++) {
        const int64_t *r = H->h_ranges + 3 * out_first[s];
        for (int k = 0; k < H->h_counts[s]; k++) {
            AfskRxStreamEvent v;
            v.stream = s; v.recorded = (int32_t)r[3 * k]; v.call = H->calls[s] + k; v.start = r[3 * k + 1]; v.end = r[3 * k + 2];
            H->ev.push_back(v);
            if (!v.recorded) {
                src.push_back(-1);
            } else if (k == 0 && H->pending[s] == v.start && H->pclock[s] >= 0) {
                fch[s] = nf;
                fev.push_back((int)H->ev.size() - 1);
                src.push_back(-2 - nf++);
            } else {
                src.push_back((int)H->rec_start.size());
                // (a recording whose samples were not kept is one decided from its length and baud alone)
                H->rec_start.push_back(v.start < H->keep[s] ? 0 : A.off[s] + v.start - A.base[s]);
                H->rec_len.push_back(v.end - v.start);
                H->rec_baud.push_back(H->baud[s]);
                H->rec_amp_end.push_back(H->params[s].amp_end);
            }
        }
    }
    // the recordings pending after this push; clocks of those that reached 4096 frames
    std::vector<int64_t> R(S), clk(S), dec(S, 0), pw0(S, 0), pw_np(S);
    std::vector<uint8_t> stored(S, 0);             // the recording was pending with its clock stored, and still is
    std::vector<int> cch;
    uint32_t qmask = 0;
    int nq[7] = {0};
    for (int s = 0; s < S; s++) {
        const GateState &g = H->h_state[s];
        R[s] = g.phase == 2 ? g.mark * C : -1;
        const bool same = R[s] >= 0 && R[s] == H->pending[s];
        stored[s] = same && H->pclock[s] >= 0;
        clk[s] = same ? H->pclock[s] : -1;
        const int bf = bits_bf(H->baud[s]);
        if (R[s] >= 0 && clk[s] < 0 && bf > 0 && H->np[s] - R[s] >= AFSK_SYNC_FRAMES) {
            const int c = (int)cch.size();
            ccap[c] = CapDesc{A.off[s] + R[s] - A.base[s], H->np[s] - R[s], 0, 0, bf, 0, 0, 0};
            cch.push_back(s);
            if (bf >= 8 && bf <= 24) nq[bf / 4]++;
        }
    }
    const int nc = (int)cch.size();
    if (nc > 0) {
        int qo[7] = {0};
        for (int q = 2, o = 0; q <= 6; q++) { qo[q] = o; o += nq[q]; }
        int qn[7] = {0};
        for (int c = 0; c < nc; c++)
            if (ccap[c].bf >= 8 && ccap[c].bf <= 24) { const int q = ccap[c].bf / 4; cq[qo[q] + qn[q]++] = c; }
        AFSK_CUDA(cudaMemcpyAsync(H->d_bdesc, hb, H->o_clk, cudaMemcpyHostToDevice, st));
        const CapDesc *d_ccap = reinterpret_cast<const CapDesc *>(db + H->o_ccap);
        const int32_t *d_cq = reinterpret_cast<const int32_t *>(db + H->o_cq);
        int32_t *d_clk = reinterpret_cast<int32_t *>(H->d_bdesc + H->o_clk);
        int nqc = 0;
        for (int q = 2; q <= 6; q++) {
            if (!nq[q]) continue;
            switch (q) {
            case 2: k_clock_q<2><<<nq[q], kClockThreads, 0, st>>>(x, d_ccap, d_cq + qo[q], d_clk); break;
            case 3: k_clock_q<3><<<nq[q], kClockThreads, 0, st>>>(x, d_ccap, d_cq + qo[q], d_clk); break;
            case 4: k_clock_q<4><<<nq[q], kClockThreads, 0, st>>>(x, d_ccap, d_cq + qo[q], d_clk); break;
            case 5: k_clock_q<5><<<nq[q], kClockThreads, 0, st>>>(x, d_ccap, d_cq + qo[q], d_clk); break;
            default: k_clock_q<6><<<nq[q], kClockThreads, 0, st>>>(x, d_ccap, d_cq + qo[q], d_clk); break;
            }
            qmask |= 1u << q;
            nqc += nq[q];
            H->n_launches++;
        }
        // (no capture here has a status of its own: k_clock writes no result)
        if (nqc < nc) {
            k_clock<<<nc, kClockThreads, 0, st>>>(x, d_ccap, d_clk, H->d_fres, qmask);
            H->n_launches++;
        }
        AFSK_CUDA(cudaGetLastError());
        AFSK_CUDA(cudaMemcpyAsync(h_clk, d_clk, sizeof(int32_t) * nc, cudaMemcpyDeviceToHost, st));
        AFSK_CUDA(cudaStreamSynchronize(st));
        for (int c = 0; c < nc; c++) clk[cch[c]] = h_clk[c];
    }
    // windows decided after this push, and the end of every channel's plane stream (a final recording's words first).
    // Payload mode: fin_ended / ended, the final / pending recording's result was fixed by the last push (h_fst).
    std::vector<int64_t> K(S, 0);
    std::vector<uint8_t> fin_ended(S, 0), ended(S, 0);
    for (int s = 0; s < S; s++) {
        int64_t e = H->pw_pushed[s];
        fin_ended[s] = pmode && fch[s] >= 0 && H->h_fst[s].phase == 2;
        ended[s] = pmode && stored[s] && H->h_fst[s].phase == 2;
        if (fch[s] >= 0) {
            const AfskRxStreamEvent &v = H->ev[fev[fch[s]]];
            K[s] = windows_of(v.end - v.start, bits_bf(H->baud[s]), H->pclock[s]);
            if (!fin_ended[s]) e = std::max(e, H->pw_rec[s] + 4 * ((K[s] + 31) / 32));
        }
        if (R[s] >= 0 && clk[s] >= 0) {
            const int bf = bits_bf(H->baud[s]);
            const int64_t span = H->np[s] - R[s] - clk[s];
            dec[s] = ended[s] ? H->pdecided[s] : span > 0 ? (span / bf) & ~(int64_t)31 : 0;
            pw0[s] = stored[s] ? H->pw_rec[s] : e;
            e = std::max(e, pw0[s] + 4 * (dec[s] / 32));
        }
        pw_np[s] = e;
    }
    int npm = 0;
    bool pcompact = false;
    cudaError_t err = slots_retain(Pl, S, H->pw_pushed.data(), pw_np.data(), H->pw_keep.data(), H->new_off.data(), H->new_cap.data(),
                                   seg_pmov, tf_pmov, npm, pcompact);
    if (err != cudaSuccess) return streams_fail(err);
    // payload mode: the windows each pending recording is framed up to (those of the chunks the gate has walked, which
    // every later end of the recording includes, as far as they are decided), and the end of every channel's payload
    // stream with room for every byte its frame jobs can write (a final recording's bytes first)
    std::vector<int64_t> kend(S, 0), py0(S, 0), py_np(S, 0);
    int nym = 0;
    bool ycompact = false;
    if (pmode) {
        const FrameState fresh = {0, 0, 0, 0, 0, {0, 0, 0}};
        auto room = [](const FrameState &f, int64_t k) {          // samples, after framing up to window k
            const int64_t b = f.phase == 2 ? f.nbytes
                                           : ((f.phase == 1 ? f.consumed - f.k0 : 0) + std::max<int64_t>(k - f.consumed, 0)) / 14 + 1;
            return (b + 1) / 2;
        };
        for (int s = 0; s < S; s++) {
            const GateState &g = H->h_state[s];
            int64_t e = H->py_pushed[s];
            if (fch[s] >= 0) e = std::max(e, H->py_rec[s] + room(H->h_fst[s], K[s]));
            if (R[s] >= 0 && clk[s] >= 0) {
                if (!ended[s]) kend[s] = std::min(windows_of((g.pos - g.mark) * C, bits_bf(H->baud[s]), clk[s]), dec[s]);
                py0[s] = stored[s] ? H->py_rec[s] : e;
                e = std::max(e, py0[s] + room(stored[s] ? H->h_fst[s] : fresh, kend[s]));
            }
            py_np[s] = e;
        }
        err = slots_retain(Y, S, H->py_pushed.data(), py_np.data(), H->py_keep.data(), H->new_off.data(), H->new_cap.data(), seg_ymov,
                           tf_ymov, nym, ycompact);
        if (err != cudaSuccess) return streams_fail(err);
    }
    // window jobs (word positions after the moves), frame captures and frame jobs
    auto word_at = [&](int s, int64_t pw) { return (Pl.off[s] + pw - Pl.base[s]) / 4; };
    auto byte_at = [&](int s, int64_t py) { return 2 * (Y.off[s] + py - Y.base[s]); };
    int nw = 0;
    tf_win[0] = 0;
    auto add_job = [&](int s, int64_t x0, int64_t w0, int64_t nwin) {
        const int bf = bits_bf(H->baud[s]);
        win[nw] = WinJob{x0, w0, (int32_t)nwin, bf, clamp_thr(H->params[s].amp_end) * bf, 0};
        tf_win[nw + 1] = tf_win[nw] + ((nwin + 31) / 32 + kWinTileWords - 1) / kWinTileWords;
        nw++;
    };
    int64_t fo = 0, fmax = 0, fsum = 0;
    int nj = 0;
    for (int s = 0; s < S; s++) {
        const int bf = bits_bf(H->baud[s]);
        const bool frame_new = pmode && kend[s] > (stored[s] ? H->h_fst[s].consumed : 0);
        if (fch[s] >= 0) {
            const int j = fch[s];
            const AfskRxStreamEvent &v = H->ev[fev[j]];
            const int64_t k0 = H->pdecided[s], n = v.end - v.start;
            if (K[s] > k0 && !fin_ended[s])
                add_job(s, A.off[s] + v.start + H->pclock[s] + k0 * bf - A.base[s], word_at(s, H->pw_rec[s]) + k0 / 32, K[s] - k0);
            fcap[j] = CapDesc{0, n, word_at(s, H->pw_rec[s]), fo, bf, clamp_thr(H->params[s].amp_end), 0, 0};
            fclk[j] = (int32_t)H->pclock[s];
            if (pmode)
                fjob[nj++] = FrameJob{H->h_fst[s], word_at(s, H->pw_rec[s]), K[s], byte_at(s, H->py_rec[s]), fo, s,
                                      kFrFinal | (frame_new ? kFrKeepState : 0), (int32_t)H->pclock[s], bf, j, {0, 0, 0}};
            const int64_t kmax = (n - bf + bf - 1) / bf;
            fo += (kmax / 14 + 16 + 15) & ~(int64_t)15;
            fmax = std::max(fmax, kmax);
            fsum += kmax;
        }
        const int64_t d0 = stored[s] ? H->pdecided[s] : 0;
        if (R[s] >= 0 && clk[s] >= 0 && dec[s] > d0)
            add_job(s, A.off[s] + R[s] + clk[s] + d0 * bf - A.base[s], word_at(s, pw0[s]) + d0 / 32, dec[s] - d0);
        if (frame_new)
            fjob[nj++] = FrameJob{stored[s] ? H->h_fst[s] : FrameState{}, word_at(s, pw0[s]), kend[s], byte_at(s, py0[s]), 0, s, 0,
                                  (int32_t)clk[s], bf, 0, {0, 0, 0}};
    }
    const size_t fres_bytes = sizeof(AfskRxResult) * (size_t)nf;
    if (nf > 0) {
        err = grow_device((void **)&H->d_fout, &H->fout_cap, (size_t)fo);
        if (err == cudaSuccess) err = grow_device((void **)&H->d_fres, &H->fres_cap, fres_bytes);
        if (err == cudaSuccess) err = grow_pinned((void **)&H->h_fdec, &H->h_fdec_cap, fres_bytes + (size_t)fo);
        if (err != cudaSuccess) return streams_fail(err);
    }
    if (npm > 0 || nw > 0 || nf > 0 || nym > 0 || nj > 0)
        AFSK_CUDA(cudaMemcpyAsync(H->d_bdesc + H->o_seg_pmov, hb + H->o_seg_pmov, H->bdesc_bytes - H->o_seg_pmov, cudaMemcpyHostToDevice, st));
    slots_move(Pl, pcompact, npm, db + H->o_seg_pmov, db + H->o_tf_pmov, tf_pmov[npm], st, H->n_launches);
    if (pmode) slots_move(Y, ycompact, nym, db + H->o_seg_ymov, db + H->o_tf_ymov, tf_ymov[nym], st, H->n_launches);
    uint2 *planes = reinterpret_cast<uint2 *>(Pl.arena[Pl.cur]);
    if (nw > 0) {
        k_stream_windows<<<(unsigned)tf_win[nw], 32 * kWinWarps, 0, st>>>(x, planes, reinterpret_cast<const WinJob *>(db + H->o_win),
                                                                         reinterpret_cast<const int64_t *>(db + H->o_tf_win), nw);
        H->n_launches++;
    }
    if (nj > 0) {
        k_stream_frame<<<(unsigned)((nj + kStreamFrameWarps - 1) / kStreamFrameWarps), 32 * kStreamFrameWarps, 0, st>>>(
            planes, reinterpret_cast<uint8_t *>(Y.arena[Y.cur]), H->d_fst, reinterpret_cast<const FrameJob *>(db + H->o_fjob), H->d_fout,
            H->d_fres, nj);
        H->n_launches++;
        AFSK_CUDA(cudaGetLastError());
        AFSK_CUDA(cudaMemcpyAsync(H->h_fst, H->d_fst, sizeof(FrameState) * S, cudaMemcpyDeviceToHost, st));
    } else if (nf > 0) {
        launch_frame(0, nf, reinterpret_cast<const CapDesc *>(db + H->o_fcap), reinterpret_cast<const int32_t *>(db + H->o_fclk), planes,
                     H->d_fout, H->d_fres, fmax, fsum, nf, st);
        H->n_launches++;
    }
    if (nf > 0) {
        AFSK_CUDA(cudaGetLastError());
        AFSK_CUDA(cudaMemcpyAsync(H->h_fdec, H->d_fres, fres_bytes, cudaMemcpyDeviceToHost, st));
        AFSK_CUDA(cudaMemcpyAsync(H->h_fdec + fres_bytes, H->d_fout, (size_t)fo, cudaMemcpyDeviceToHost, st));
    }
    AFSK_CUDA(cudaGetLastError());
    const AfskRxResult *rr = nullptr;
    const int64_t *oo = nullptr;
    size_t res_bytes = 0;
    if (!H->rec_start.empty()) {
        const int rc = streams_decode_plan(H, x, st, &rr, &oo, &res_bytes);
        if (rc != AFSK_OK) return rc;
    } else {
        AFSK_CUDA(cudaStreamSynchronize(st));
    }
    // results and payloads in event order
    const int nev = (int)H->ev.size();
    const AfskRxResult *fr = reinterpret_cast<const AfskRxResult *>(H->h_fdec);
    H->res.assign((size_t)nev, AfskRxResult{0, -1, -1, 0, 0});
    H->payload_off.assign((size_t)nev + 1, 0);
    H->payload.clear();
    for (int i = 0; i < nev; i++) {
        H->payload_off[i] = (int64_t)H->payload.size();
        if (src[i] == -1) continue;
        const uint8_t *p;
        if (src[i] >= 0) {
            H->res[i] = rr[src[i]];
            p = H->h_dec + res_bytes + oo[src[i]];
        } else {
            const int j = -2 - src[i];
            H->res[i] = fr[j];
            p = H->h_fdec + fres_bytes + fcap[j].out_off;
        }
        if (H->res[i].nbytes > 0) H->payload.insert(H->payload.end(), p, p + H->res[i].nbytes);
    }
    H->payload_off[nev] = (int64_t)H->payload.size();
    // the channels' new state
    for (int s = 0; s < S; s++) {
        const GateState &g = H->h_state[s];
        const int bf = bits_bf(H->baud[s]);
        H->calls[s] = g.call;
        H->pushed[s] = H->np[s];
        H->pending[s] = R[s];
        const bool planes_on = R[s] >= 0 && clk[s] >= 0;
        // payload mode: what the pending recording's framing still needs (h_fst as this push left it)
        const FrameState f = pmode ? H->h_fst[s] : FrameState{};
        const bool fixed = pmode && planes_on && f.phase == 2;
        const int64_t need = !pmode ? 0 : f.phase == 1 ? f.k0 + 14 * f.nbytes : std::max<int64_t>(f.consumed - 3, 0);
        H->keep[s] = R[s] < 0 || bf == 0 || fixed ? g.pos * C
                     : planes_on                  ? std::min<int64_t>(g.pos * C, R[s] + clk[s] + dec[s] * bf)
                                                  : R[s];
        H->pclock[s] = planes_on ? clk[s] : -1;
        H->pdecided[s] = planes_on ? dec[s] : 0;
        H->pw_rec[s] = planes_on ? pw0[s] : 0;
        H->pw_pushed[s] = pw_np[s];
        H->pw_keep[s] = planes_on && !fixed ? pw0[s] + 4 * (need / 32) : pw_np[s];
        if (pmode) {
            H->py_rec[s] = planes_on ? py0[s] : 0;
            H->py_pushed[s] = py_np[s];
            H->py_keep[s] = planes_on ? py0[s] : py_np[s];
        }
    }
    return AFSK_OK;
}

// a push or finish with valid arguments: any failure may leave the channels between two states, so the
// handle refuses every later push / finish
static int streams_call(AfskRxStreams *H, const void *samples, int on_device, const int64_t *off, int64_t inter, int format,
                        int64_t pitch, void *stream,
                        const uint8_t *fin, const int32_t *new_baud, const GateParams *new_params, int64_t *n_events)
{
    if (H->failed) { afsk_set_error("afsk_rx_streams: an earlier push failed; destroy the handle"); return AFSK_E_CUDA; }
    AfskDeviceGuard guard(H->device);
    if (!guard.ok) { afsk_set_error("cannot select device %d", H->device); return AFSK_E_CUDA; }
    if (H->retain != AFSK_RETAIN_SAMPLES && !fin) {
        // a window range of one push (WinJob.nwin) spans the piece plus a tail of under 33 bit lengths: below 2^31 windows
        for (int s = 0; s < H->S; s++)
            if ((inter >= 0 ? inter : off[s + 1] - off[s]) > kBitsMaxPiece) {
                afsk_set_error("afsk_rx_streams: bits and payload retention take at most 2^32 frames per channel and push (channel %d)", s);
                return AFSK_E_ARG;
            }
    }
    H->used = true;
    const int rc = streams_run(H, samples, on_device, off, inter, format, pitch, (cudaStream_t)stream, fin, new_baud, new_params, n_events);
    if (rc != AFSK_OK) {
        H->failed = true;
        H->ev.clear(); H->res.clear(); H->payload.clear(); H->payload_off.clear();
    }
    return rc;
}

// checks one channel's settings: AFSK_E_ARG for a negative timeout, AFSK_E_BAUD where the reference
// constructor raises
static int rx_settings_check(const char *fn, int s, int baud, int64_t timeout_frames)
{
    if (timeout_frames < 0) { afsk_set_error("%s: negative timeout on channel %d", fn, s); return AFSK_E_ARG; }
    int bf, ml, sl;
    if (!afsk_tone_geometry(baud, &bf, &ml, &sl)) { afsk_set_error("Invalid baud rate. (%s: channel %d, baud %d)", fn, s, baud); return AFSK_E_BAUD; }
    return AFSK_OK;
}

// the bits- and payload-mode buffers of a handle (set_retention): freed when the handle changes its mode
static void streams_free_bits(AfskRxStreams *H)
{
    for (void *p : {(void *)H->pln.arena[0], (void *)H->pln.arena[1], (void *)H->d_bdesc, (void *)H->d_fout, (void *)H->d_fres,
                    (void *)H->pay.arena[0], (void *)H->pay.arena[1], (void *)H->d_fst})
        cudaFree(p);
    for (void *p : {(void *)H->h_bdesc, (void *)H->h_fdec, (void *)H->h_fst})
        if (p) cudaFreeHost(p);
    H->pln.arena[0] = H->pln.arena[1] = H->pay.arena[0] = H->pay.arena[1] = nullptr;
    H->pln.arena_cap[0] = H->pln.arena_cap[1] = H->pay.arena_cap[0] = H->pay.arena_cap[1] = 0;
    H->d_bdesc = H->h_bdesc = H->d_fout = H->h_fdec = nullptr;
    H->d_fres = nullptr;
    H->d_fst = H->h_fst = nullptr;
    H->bdesc_bytes = H->fout_cap = H->fres_cap = H->h_fdec_cap = 0;
}

int afsk_rx_streams_create_each(int device, int S, const int32_t *h_baud, const int32_t *h_amp_start, const int32_t *h_amp_end,
                                const int64_t *h_timeout_frames, AfskRxStreams **h)
{
    if (!h || S < 1 || !h_baud || !h_amp_start || !h_amp_end || !h_timeout_frames) {
        afsk_set_error("afsk_rx_streams_create_each: bad argument (S >= 1, non-null arrays)");
        return AFSK_E_ARG;
    }
    for (int s = 0; s < S; s++) {
        const int rc = rx_settings_check("afsk_rx_streams_create_each", s, h_baud[s], h_timeout_frames[s]);
        if (rc != AFSK_OK) return rc;
    }
    AfskDeviceGuard guard(device);
    if (!guard.ok) { afsk_set_error("cannot select device %d", device); return AFSK_E_CUDA; }
    AfskRxStreams *H = new (std::nothrow) AfskRxStreams();
    if (!H) return AFSK_E_ARG;
    H->device = device; H->S = S;
    H->baud.assign(h_baud, h_baud + S);
    H->params.resize((size_t)S);
    for (int s = 0; s < S; s++) H->params[s] = GateParams{h_amp_start[s], h_amp_end[s], h_timeout_frames[s]};
    for (auto *v : {&H->pushed, &H->keep, &H->calls, &H->smp.off, &H->smp.cap, &H->smp.base, &H->np, &H->new_off, &H->new_cap,
                    &H->pdecided, &H->pw_rec, &H->pw_pushed, &H->pw_keep, &H->pln.off, &H->pln.cap, &H->pln.base, &H->py_rec,
                    &H->py_pushed, &H->py_keep, &H->pay.off, &H->pay.cap, &H->pay.base})
        v->assign((size_t)S, 0);
    H->pending.assign((size_t)S, -1);
    H->pclock.assign((size_t)S, -1);
    size_t o = 0;
    auto carve = [&](size_t bytes) { const size_t at = o; o += (bytes + 15) & ~(size_t)15; return at; };
    H->o_seg_app = carve(sizeof(CopySeg) * S); H->o_tf_app = carve(8 * ((size_t)S + 1));
    H->o_seg_mov = carve(sizeof(CopySeg) * S); H->o_tf_mov = carve(8 * ((size_t)S + 1));
    H->o_first = carve(8 * ((size_t)S + 1)); H->o_amp_off = carve(8 * (size_t)S); H->o_out_first = carve(8 * (size_t)S);
    H->o_fin = carve((size_t)S);
    H->desc_bytes = o;
    cudaError_t e = cudaMalloc((void **)&H->d_desc, H->desc_bytes);
    if (e == cudaSuccess) e = cudaMallocHost((void **)&H->h_desc, H->desc_bytes);
    if (e == cudaSuccess) e = cudaMalloc((void **)&H->d_state, sizeof(GateState) * S);
    if (e == cudaSuccess) e = cudaMallocHost((void **)&H->h_state, sizeof(GateState) * S);
    if (e == cudaSuccess) e = cudaMalloc((void **)&H->d_counts, sizeof(int32_t) * S);
    if (e == cudaSuccess) e = cudaMallocHost((void **)&H->h_counts, sizeof(int32_t) * S);
    if (e == cudaSuccess) e = cudaMalloc((void **)&H->d_params, sizeof(GateParams) * S);
    if (e == cudaSuccess) e = cudaMemcpy(H->d_params, H->params.data(), sizeof(GateParams) * S, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(H->d_state, 0, sizeof(GateState) * S);
    if (e != cudaSuccess) {
        afsk_rx_streams_destroy(H);
        return streams_fail(e);
    }
    *h = H;
    return AFSK_OK;
}

int afsk_rx_streams_create(int device, int S, int baud, int amp_start, int amp_end, int64_t timeout_frames, AfskRxStreams **h)
{
    const size_t n = S > 0 ? (size_t)S : 1;
    const std::vector<int32_t> b(n, baud), a0(n, amp_start), a1(n, amp_end);
    const std::vector<int64_t> t(n, timeout_frames < 0 ? 0 : timeout_frames);     // any timeout <= 0 gates alike
    return afsk_rx_streams_create_each(device, S, b.data(), a0.data(), a1.data(), t.data(), h);
}

int afsk_rx_streams_set_retention(AfskRxStreams *H, int mode)
{
    const char *fn = "afsk_rx_streams_set_retention";
    if (!H || (mode != AFSK_RETAIN_SAMPLES && mode != AFSK_RETAIN_BITS && mode != AFSK_RETAIN_PAYLOAD)) {
        afsk_set_error("%s: bad argument", fn);
        return AFSK_E_ARG;
    }
    if (H->used) { afsk_set_error("%s: the retention mode is chosen before the first push or finish", fn); return AFSK_E_ARG; }
    AfskDeviceGuard guard(H->device);
    if (!guard.ok) { afsk_set_error("cannot select device %d", H->device); return AFSK_E_CUDA; }
    streams_free_bits(H);
    if (mode != AFSK_RETAIN_SAMPLES) {
        const size_t S = (size_t)H->S;
        size_t o = 0;
        auto carve = [&](size_t bytes) { const size_t at = o; o += (bytes + 15) & ~(size_t)15; return at; };
        // (the clock part comes first: the clock launches copy the block up to o_clk only)
        H->o_ccap = carve(sizeof(CapDesc) * S); H->o_cq = carve(sizeof(int32_t) * S); H->o_clk = carve(sizeof(int32_t) * S);
        H->o_seg_pmov = carve(sizeof(CopySeg) * S); H->o_tf_pmov = carve(8 * (S + 1));
        H->o_win = carve(sizeof(WinJob) * 2 * S); H->o_tf_win = carve(8 * (2 * S + 1));   // a final tail and a new recording per channel
        H->o_fcap = carve(sizeof(CapDesc) * S); H->o_fclk = carve(sizeof(int32_t) * S);
        if (mode == AFSK_RETAIN_PAYLOAD) {
            H->o_seg_ymov = carve(sizeof(CopySeg) * S); H->o_tf_ymov = carve(8 * (S + 1));
            H->o_fjob = carve(sizeof(FrameJob) * 2 * S);                                      // a final and a pending recording per channel
        }
        H->bdesc_bytes = o;
        cudaError_t e = cudaMalloc((void **)&H->d_bdesc, o);
        if (e == cudaSuccess) e = cudaMallocHost((void **)&H->h_bdesc, o);
        if (e == cudaSuccess && mode == AFSK_RETAIN_PAYLOAD) {
            e = cudaMalloc((void **)&H->d_fst, sizeof(FrameState) * S);
            if (e == cudaSuccess) e = cudaMallocHost((void **)&H->h_fst, sizeof(FrameState) * S);
            if (e == cudaSuccess) e = cudaMemset(H->d_fst, 0, sizeof(FrameState) * S);
            if (e == cudaSuccess) memset(H->h_fst, 0, sizeof(FrameState) * S);
        }
        if (e != cudaSuccess) {
            streams_free_bits(H);
            return streams_fail(e);
        }
    }
    H->retain = mode;
    return AFSK_OK;
}

int afsk_rx_streams_push(AfskRxStreams *H, const int16_t *samples, int on_device, const int64_t *h_offsets, void *stream,
                         int64_t *n_events)
{
    if (!H || !h_offsets || !n_events) { afsk_set_error("afsk_rx_streams_push: null argument"); return AFSK_E_ARG; }
    if (h_offsets[0] < 0) { afsk_set_error("afsk_rx_streams_push: negative offset"); return AFSK_E_ARG; }
    for (int s = 0; s < H->S; s++)
        if (h_offsets[s + 1] < h_offsets[s]) { afsk_set_error("afsk_rx_streams_push: offsets decrease at channel %d", s); return AFSK_E_ARG; }
    if (h_offsets[H->S] > h_offsets[0] && !samples) { afsk_set_error("afsk_rx_streams_push: null samples"); return AFSK_E_ARG; }
    if (on_device && (reinterpret_cast<uintptr_t>(samples) & 15) != 0) {
        afsk_set_error("afsk_rx_streams_push: device samples must be 16-byte aligned");
        return AFSK_E_ARG;
    }
    return streams_call(H, samples, on_device, h_offsets, -1, AFSK_SAMPLE_S16, 0, stream, nullptr, nullptr, nullptr, n_events);
}

// the argument checks of an interleaved push (fn names the entry point in the error)
static int push_frames_check(const char *fn, AfskRxStreams *H, const void *frames, int format, int64_t n_frames, int64_t row_pitch,
                             int64_t *n_events)
{
    if (!H || !n_events || n_frames < 0 || (n_frames > 0 && !frames)) { afsk_set_error("%s: bad argument", fn); return AFSK_E_ARG; }
    const int size = afsk_sample_size(format);
    if (!size) { afsk_set_error("%s: unknown sample format %d", fn, format); return AFSK_E_ARG; }
    if (row_pitch < H->S) { afsk_set_error("%s: row_pitch %lld < S = %d", fn, (long long)row_pitch, H->S); return AFSK_E_ARG; }
    if ((reinterpret_cast<uintptr_t>(frames) & (uintptr_t)(size - 1)) != 0) {
        afsk_set_error("%s: frames must be aligned to the sample size (%d bytes)", fn, size);
        return AFSK_E_ARG;
    }
    if (n_frames > (INT64_MAX / 16) / row_pitch) { afsk_set_error("%s: row_pitch * n_frames overflows", fn); return AFSK_E_ARG; }
    if ((int64_t)((H->S + kDiC - 1) / kDiC) * ((n_frames + kDiF + kDiHalo - 1) / kDiF) > 0x7FFFFFFFLL) {
        afsk_set_error("%s: piece too large", fn);
        return AFSK_E_ARG;
    }
    return AFSK_OK;
}

int afsk_rx_streams_push_interleaved(AfskRxStreams *H, const int16_t *frames, int on_device, int64_t n_frames, void *stream,
                                     int64_t *n_events)
{
    const char *fn = "afsk_rx_streams_push_interleaved";
    const int rc = push_frames_check(fn, H, frames, AFSK_SAMPLE_S16, n_frames, H ? H->S : 0, n_events);
    if (rc != AFSK_OK) return rc;
    if (on_device && (reinterpret_cast<uintptr_t>(frames) & 15) != 0) {
        afsk_set_error("%s: device frames must be 16-byte aligned", fn);
        return AFSK_E_ARG;
    }
    return streams_call(H, frames, on_device, nullptr, n_frames, AFSK_SAMPLE_S16, H->S, stream, nullptr, nullptr, nullptr, n_events);
}

int afsk_rx_streams_push_frames(AfskRxStreams *H, const void *frames, int format, int on_device, int64_t n_frames, int64_t row_pitch,
                                void *stream, int64_t *n_events)
{
    const int rc = push_frames_check("afsk_rx_streams_push_frames", H, frames, format, n_frames, row_pitch, n_events);
    if (rc != AFSK_OK) return rc;
    return streams_call(H, frames, on_device, nullptr, n_frames, format, row_pitch, stream, nullptr, nullptr, nullptr, n_events);
}

int afsk_rx_streams_finish_some(AfskRxStreams *H, int n, const int32_t *h_streams, const int32_t *h_baud, const int32_t *h_amp_start,
                                const int32_t *h_amp_end, const int64_t *h_timeout_frames, void *stream, int64_t *n_events)
{
    const char *fn = "afsk_rx_streams_finish_some";
    if (!H || !n_events || n < 0 || n > H->S || (n > 0 && !h_streams)) { afsk_set_error("%s: bad argument", fn); return AFSK_E_ARG; }
    const int given = (h_baud != nullptr) + (h_amp_start != nullptr) + (h_amp_end != nullptr) + (h_timeout_frames != nullptr);
    if (given != 0 && given != 4) { afsk_set_error("%s: the settings arrays are all given or all NULL", fn); return AFSK_E_ARG; }
    std::vector<uint8_t> fin((size_t)H->S, 0);
    for (int i = 0; i < n; i++) {
        const int s = h_streams[i];
        if (s < 0 || s >= H->S) { afsk_set_error("%s: stream %d out of range", fn, s); return AFSK_E_ARG; }
        if (fin[s]) { afsk_set_error("%s: stream %d listed twice", fn, s); return AFSK_E_ARG; }
        fin[s] = 1;
    }
    if (!given) return streams_call(H, nullptr, 0, nullptr, -1, AFSK_SAMPLE_S16, 0, stream, fin.data(), nullptr, nullptr, n_events);
    for (int i = 0; i < n; i++) {
        const int rc = rx_settings_check(fn, h_streams[i], h_baud[i], h_timeout_frames[i]);
        if (rc != AFSK_OK) return rc;
    }
    std::vector<int32_t> baud = H->baud;
    std::vector<GateParams> params = H->params;
    for (int i = 0; i < n; i++) {
        baud[h_streams[i]] = h_baud[i];
        params[h_streams[i]] = GateParams{h_amp_start[i], h_amp_end[i], h_timeout_frames[i]};
    }
    return streams_call(H, nullptr, 0, nullptr, -1, AFSK_SAMPLE_S16, 0, stream, fin.data(), baud.data(), params.data(), n_events);
}

int afsk_rx_streams_finish(AfskRxStreams *H, void *stream, int64_t *n_events)
{
    if (!H || !n_events) { afsk_set_error("afsk_rx_streams_finish: null argument"); return AFSK_E_ARG; }
    std::vector<int32_t> all((size_t)H->S);
    for (int s = 0; s < H->S; s++) all[s] = s;
    return afsk_rx_streams_finish_some(H, H->S, all.data(), nullptr, nullptr, nullptr, nullptr, stream, n_events);
}

int afsk_rx_streams_events(const AfskRxStreams *H, const AfskRxStreamEvent **ev, const AfskRxResult **res, const uint8_t **payload,
                           const int64_t **payload_off)
{
    if (!H) return AFSK_E_ARG;
    if (ev) *ev = H->ev.data();
    if (res) *res = H->res.data();
    if (payload) *payload = H->payload.data();
    if (payload_off) *payload_off = H->payload_off.empty() ? nullptr : H->payload_off.data();
    return AFSK_OK;
}

int afsk_rx_streams_state(const AfskRxStreams *H, int s, int64_t *pushed, int64_t *pending_start, int64_t *retained)
{
    if (!H || s < 0 || s >= H->S) { afsk_set_error("afsk_rx_streams_state: bad argument"); return AFSK_E_ARG; }
    if (pushed) *pushed = H->pushed[s];
    if (pending_start) *pending_start = H->pending[s];
    if (retained) *retained = H->pushed[s] - H->keep[s];
    return AFSK_OK;
}

int afsk_rx_streams_pending_bits(const AfskRxStreams *H, int s, int32_t *clock, int64_t *windows)
{
    if (!H || s < 0 || s >= H->S) { afsk_set_error("afsk_rx_streams_pending_bits: bad argument"); return AFSK_E_ARG; }
    if (clock) *clock = H->pending[s] >= 0 ? (int32_t)H->pclock[s] : -1;
    if (windows) *windows = H->pending[s] >= 0 ? H->pdecided[s] : 0;
    return AFSK_OK;
}

int afsk_rx_streams_pending_planes(const AfskRxStreams *H, int s, const uint32_t **d_planes, int64_t *first_window, int64_t *n_windows)
{
    if (!H || s < 0 || s >= H->S || !d_planes || !first_window || !n_windows) {
        afsk_set_error("afsk_rx_streams_pending_planes: bad argument");
        return AFSK_E_ARG;
    }
    *d_planes = nullptr; *first_window = 0; *n_windows = 0;
    if (H->retain == AFSK_RETAIN_SAMPLES || H->pending[s] < 0 || H->pclock[s] < 0) return AFSK_OK;
    // plane positions count four samples per word: the recording's word 0 is at pw_rec, the channel keeps from pw_keep
    const int64_t base = (H->pw_keep[s] - H->pw_rec[s]) / 4;
    const int64_t n = H->pdecided[s] - 32 * base;
    if (n <= 0) return AFSK_OK;
    const Slots &Pl = H->pln;
    *d_planes = reinterpret_cast<const uint32_t *>(reinterpret_cast<const uint2 *>(Pl.arena[Pl.cur]) + (Pl.off[s] + H->pw_keep[s] - Pl.base[s]) / 4);
    *first_window = 32 * base;
    *n_windows = n;
    return AFSK_OK;
}

int afsk_rx_streams_arena_bytes(const AfskRxStreams *H, int64_t *bytes)
{
    if (!H || !bytes) return AFSK_E_ARG;
    *bytes = (int64_t)(H->smp.arena_cap[0] + H->smp.arena_cap[1] + H->stage_cap + H->desc_bytes + H->amp_cap + H->ranges_cap + H->out_cap +
                       H->res_cap + (sizeof(GateState) + sizeof(int32_t) + sizeof(GateParams)) * (size_t)H->S +
                       H->pln.arena_cap[0] + H->pln.arena_cap[1] + H->bdesc_bytes + H->fout_cap + H->fres_cap +
                       H->pay.arena_cap[0] + H->pay.arena_cap[1] + (H->d_fst ? sizeof(FrameState) * (size_t)H->S : 0));
    return AFSK_OK;
}

int afsk_rx_streams_counters(const AfskRxStreams *H, int64_t *launches, int64_t *moved_frames, int64_t *compactions)
{
    if (!H) return AFSK_E_ARG;
    if (launches) *launches = H->n_launches;
    if (moved_frames) *moved_frames = H->smp.n_moved;
    if (compactions) *compactions = H->smp.n_compactions;
    return AFSK_OK;
}

int afsk_rx_streams_plane_counters(const AfskRxStreams *H, int64_t *moved_words, int64_t *compactions)
{
    if (!H) { afsk_set_error("afsk_rx_streams_plane_counters: bad argument"); return AFSK_E_ARG; }
    if (moved_words) *moved_words = H->pln.n_moved / 4;
    if (compactions) *compactions = H->pln.n_compactions;
    return AFSK_OK;
}

int afsk_rx_streams_pending_payload(const AfskRxStreams *H, int s, int64_t *train_end, int64_t *nbits, int32_t *ended, uint8_t *out,
                                    int64_t cap, int64_t *nbytes)
{
    if (!H || s < 0 || s >= H->S || !train_end || !nbits || !ended || !nbytes || cap < 0 || (cap > 0 && !out)) {
        afsk_set_error("afsk_rx_streams_pending_payload: bad argument");
        return AFSK_E_ARG;
    }
    *train_end = -1; *nbits = 0; *ended = 0; *nbytes = 0;
    if (H->retain != AFSK_RETAIN_PAYLOAD || H->pending[s] < 0 || H->pclock[s] < 0) return AFSK_OK;
    const FrameState &f = H->h_fst[s];
    if (f.phase >= 1) {
        *train_end = H->pclock[s] + f.k0 * (int64_t)bits_bf(H->baud[s]);
        *nbits = (f.phase == 2 ? f.k1 : f.consumed) - f.k0;
    }
    *ended = f.phase == 2;
    *nbytes = f.nbytes;
    const int64_t n = std::min<int64_t>(cap, f.nbytes);
    if (n > 0) {
        AfskDeviceGuard guard(H->device);
        if (!guard.ok) { afsk_set_error("cannot select device %d", H->device); return AFSK_E_CUDA; }
        const Slots &Y = H->pay;
        const uint8_t *src = reinterpret_cast<const uint8_t *>(Y.arena[Y.cur]) + 2 * (Y.off[s] + H->py_rec[s] - Y.base[s]);
        AFSK_CUDA(cudaMemcpy(out, src, (size_t)n, cudaMemcpyDeviceToHost));
    }
    return AFSK_OK;
}

int afsk_rx_streams_payload_counters(const AfskRxStreams *H, int64_t *moved_bytes, int64_t *compactions)
{
    if (!H) { afsk_set_error("afsk_rx_streams_payload_counters: bad argument"); return AFSK_E_ARG; }
    if (moved_bytes) *moved_bytes = 2 * H->pay.n_moved;
    if (compactions) *compactions = H->pay.n_compactions;
    return AFSK_OK;
}

int afsk_rx_streams_destroy(AfskRxStreams *H)
{
    if (!H) return AFSK_OK;
    AfskDeviceGuard guard(H->device);
    if (H->plan) afsk_rx_plan_destroy(H->plan);
    streams_free_bits(H);
    for (void *p : {(void *)H->smp.arena[0], (void *)H->smp.arena[1], (void *)H->d_stage, (void *)H->d_desc, (void *)H->d_state,
                    (void *)H->d_counts, (void *)H->d_params, (void *)H->d_amp, (void *)H->d_ranges, (void *)H->d_out, (void *)H->d_res})
        cudaFree(p);
    for (void *p : {(void *)H->h_desc, (void *)H->h_state, (void *)H->h_counts, (void *)H->h_ranges, (void *)H->h_dec})
        if (p) cudaFreeHost(p);
    delete H;
    return AFSK_OK;
}

}  // extern "C"
