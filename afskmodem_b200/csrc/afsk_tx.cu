// afsk_tx.cu — transmitter path of libafsk_b200.so (sm_100a).
//
// Replaces Transmitter.__getFrames (afskmodem.py:452-469: __bytesToBits :446-450, ECC.encode
// :166-175, training cycles :457-458, terminator :460-462, one tone per coded bit :463-467,
// 4800 zero frames :468) followed by SoundOutput.__convertFrames (:239-244, out[n] =
// frames[n & ~1], odd trailing frame dropped) for B payloads.  Elementwise and write-bound:
// each thread produces 16-byte vectors (8 samples) with coalesced 128-bit stores; the frame
// value is recomputed from the payload byte (Hamming(7,4) codeword bit -> mark/space square
// wave phase), nothing is staged in HBM.
#include <string.h>

#include <algorithm>
#include <deque>
#include <new>
#include <vector>

#include "afsk_common.cuh"

namespace {

constexpr int kSynthThreads = 256;
constexpr int kVecPerThread = 32;
constexpr int kChunkVecs = kSynthThreads * kVecPerThread;   // 8192 vectors = 65536 samples per CTA
constexpr int kMaxSymbols = kChunkVecs * 8 / 4 + 8;         // bit symbols one chunk can touch (bf >= 4)

struct __align__(16) TxDesc {
    int64_t pay_off;      // byte offset of the payload
    int64_t pay_len;
    int64_t out_off;      // sample offset of the capture (multiple of 8)
    int64_t out_len;      // frames written by save(): (len(frames) & ~1)
    int64_t total_bits;   // training + terminator + coded bits
    int64_t ts_bits;      // 2 * ts_cycles training bits (1,0,1,0,...)
    int32_t bf;           // = space tone length
    int32_t ml;           // mark tone length: bf, or bf - 2 when bf % 4 == 2 (4800, 960, 1600, 8000, 24000 baud)
    int64_t chunk_first;  // first CTA chunk of this capture
    int64_t nib_off;      // ml != bf: offset of the capture's nibble start table (2 * pay_len + 1 entries)
    int64_t pad;
};

// Hamming(7,4) generator (ECC.__M_GENERATOR :115-123): codeword bit r of nibble v, LSB = c0
__device__ __forceinline__ uint32_t hamming74_encode(uint32_t v)
{
    const uint32_t d0 = (v >> 3) & 1u, d1 = (v >> 2) & 1u, d2 = (v >> 1) & 1u, d3 = v & 1u;
    return (d0 ^ d1 ^ d3) | ((d0 ^ d2 ^ d3) << 1) | (d0 << 2) | ((d1 ^ d2 ^ d3) << 3) | (d1 << 4) | (d2 << 5) |
           (d3 << 6);
}

// bit b of the transmitted sequence (__getFrames :452-469)
__device__ __forceinline__ uint32_t tx_bit(long long b, const TxDesc &d, const uint8_t *__restrict__ pay)
{
    if (b < d.ts_bits) return (uint32_t)(~b & 1);            // training cycle = mark, space  :457-458
    const long long t = b - d.ts_bits;
    if (t < 4) return t == 0 ? 1u : 0u;                      // terminator mark, space x3     :460-462
    const long long j = t - 4;                               // coded bit index
    long long g;                                             // nibble index, high nibble first :446-450
    uint32_t r;
    if (j < 0x7FFFFFFFLL) {                                  // 32-bit divide for all but > 150 MB payloads
        const uint32_t g32 = (uint32_t)j / 7u;
        r = (uint32_t)j - 7u * g32;
        g = g32;
    } else {
        g = j / 7;
        r = (uint32_t)(j - 7 * g);
    }
    const uint32_t byte = pay[d.pay_off + (g >> 1)];
    const uint32_t nib = (g & 1) ? (byte & 15u) : (byte >> 4);
    return (hamming74_encode(nib) >> r) & 1u;
}

// frame value at phase ph of a tone (Waveforms.getSpaceTone/getMarkTone :68-85), as 2 duplicated
// int16 (SoundOutput.__convertFrames :239-244 emits every even frame twice); sym 2 = silence
__device__ __forceinline__ uint32_t tone_pair(uint32_t sym, int ph, int bf)
{
    if (sym == 2u) return 0u;
    const int q = bf >> 2, h = bf >> 1;
    bool hi;
    if (sym) hi = (ph < q) || (ph >= 2 * q && ph < 3 * q);   // mark : q HI, q LO, q HI, q LO  (q = int(bf / 4))
    else hi = ph < h;                                        // space: h HI, h LO
    return hi ? 0x7FFF7FFFu : 0x80008000u;
}

// One CTA writes 8192 consecutive 16-byte vectors of one capture.  Bits are grouped so that a group
// is a whole number of vectors (1 bit when bf % 8 == 0, else 2 bits); the CTA tabulates the vector
// patterns of every symbol combination of a group (3 or 9 combinations: space / mark / silence)
// and the bit symbols its chunk touches in shared memory, then every thread emits
// pattern[combination][vector-in-group] with one 128-bit shared load and one coalesced 128-bit store.
__global__ void __launch_bounds__(kSynthThreads) k_synth(const uint8_t *__restrict__ pay,
                                                         const TxDesc *__restrict__ descs,
                                                         const int32_t *__restrict__ chunk_cap,
                                                         int16_t *__restrict__ out)
{
    extern __shared__ __align__(16) uint8_t tx_smem[];
    const int tid = threadIdx.x;
    const long long chunk = blockIdx.x;
    const TxDesc d = descs[chunk_cap[chunk]];
    if (d.ml != d.bf) return;                                // unequal tones: k_synth_var
    const int bf = d.bf;
    const int G = (bf & 7) ? 2 : 1;                          // bits per group
    const int VG = G * bf / 8;                               // vectors per group
    const int ncomb = G == 1 ? 3 : 9;
    uint4 *tab = reinterpret_cast<uint4 *>(tx_smem);
    uint8_t *sym = tx_smem + (size_t)ncomb * VG * 16;

    const long long nvec_cap = (d.out_len + 7) >> 3;
    const long long v0 = (chunk - d.chunk_first) * kChunkVecs;
    const long long vend = min(v0 + (long long)kChunkVecs, nvec_cap);
    const long long g0 = v0 / VG, g1 = (vend - 1) / VG;
    const long long b0 = g0 * G;
    const int nb = (int)(g1 - g0 + 1) * G;
    for (int i = tid; i < nb; i += kSynthThreads) {
        const long long bi = b0 + i;
        sym[i] = bi < d.total_bits ? (uint8_t)tx_bit(bi, d, pay) : (uint8_t)2;    // 4800 zero frames :468
    }
    for (int idx = tid; idx < ncomb * VG; idx += kSynthThreads) {
        const int comb = idx / VG, k = idx - comb * VG;
        uint32_t w[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            int n = 8 * k + 2 * j;                           // even frame inside the group
            uint32_t s = (uint32_t)comb;
            if (G == 2) {
                if (n >= bf) { n -= bf; s = comb % 3; } else s = comb / 3;
            }
            w[j] = tone_pair(s, n, bf);
        }
        tab[idx] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    __syncthreads();

    uint4 *dst = reinterpret_cast<uint4 *>(out + d.out_off);
    const int vr0 = (int)(v0 - g0 * VG) + tid;               // vector index relative to group g0
    int gi = vr0 / VG, k = vr0 - gi * VG;
    const int dg = kSynthThreads / VG, dk = kSynthThreads - dg * VG;
#pragma unroll 8
    for (int r = 0; r < kVecPerThread; r++) {
        const long long vi = v0 + r * kSynthThreads + tid;
        if (vi < vend) {
            const int comb = G == 1 ? sym[gi] : sym[2 * gi] * 3 + sym[2 * gi + 1];
            dst[vi] = tab[comb * VG + k];
        }
        gi += dg; k += dk;
        if (k >= VG) { k -= VG; gi++; }
    }
}

// ------------------------------------------------------------------ unequal tone lengths ----
// When bit_frames % 4 == 2 the mark tone (two cycles of int(bf/4) HI + int(bf/4) LO, :81-85) is two
// frames shorter than the space tone, so a bit's first frame depends on how many marks precede it
// (__getFrames :463-467 just appends).  k_tx_nibscan writes the first frame of every Hamming
// codeword (exclusive scan of ones * ml + (7 - ones) * bf over the nibbles), k_synth_var locates
// each output vector's frames by binary search in that table and walks the 7 bits of the codeword.
constexpr int kScanThreads = 256;

__global__ void __launch_bounds__(kScanThreads) k_tx_nibscan(const uint8_t *__restrict__ pay,
                                                            const TxDesc *__restrict__ descs,
                                                            const int32_t *__restrict__ var_caps,
                                                            int64_t *__restrict__ nib_start)
{
    const TxDesc d = descs[var_caps[blockIdx.x]];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __shared__ long long warp_tot[kScanThreads / 32];
    int64_t *out = nib_start + d.nib_off;
    const long long G = 2 * d.pay_len;
    long long carry = 0;
    for (long long base = 0; base <= G; base += kScanThreads) {
        const long long g = base + tid;
        long long len = 0;
        if (g < G) {
            const uint32_t byte = pay[d.pay_off + (g >> 1)];
            const int ones = __popc(hamming74_encode((g & 1) ? (byte & 15u) : (byte >> 4)));
            len = (long long)ones * d.ml + (long long)(7 - ones) * d.bf;
        }
        long long inc = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) warp_tot[warp] = inc;
        __syncthreads();
        long long before = carry, total = 0;
        for (int w = 0; w < kScanThreads / 32; w++) {
            if (w < warp) before += warp_tot[w];
            total += warp_tot[w];
        }
        if (g <= G) out[g] = before + inc - len;             // exclusive: first frame of codeword g
        carry += total;
        __syncthreads();
    }
}

// Position of frame n (even) in the bit sequence of a capture with unequal tones: bit index b (training,
// terminator and coded bits counted together; b >= total_bits: the 4800 zero frames :468) and the frame's
// offset u inside that bit's tone.  One 64-bit division (training) or one binary search over the codeword
// start table (coded bits) — done once per 64 frames by k_synth_var, which then walks bit by bit.
__device__ __forceinline__ void var_locate(long long n, const TxDesc &d, const uint8_t *__restrict__ pay,
                                           const int64_t *__restrict__ ns, long long &b, int &u)
{
    const long long ml = d.ml, sl = d.bf;
    const long long T0 = (d.ts_bits >> 1) * (ml + sl);       // training cycles: mark, space  :457-458
    if (n < T0) {
        const long long cyc = n / (ml + sl);
        const long long r = n - cyc * (ml + sl);
        b = 2 * cyc + (r >= ml ? 1 : 0);
        u = (int)(r >= ml ? r - ml : r);
        return;
    }
    long long t = n - T0;
    if (t < ml) { b = d.ts_bits; u = (int)t; return; }       // terminator: mark, space x3   :460-462
    t -= ml;
    if (t < 3 * sl) { const long long k = t / sl; b = d.ts_bits + 1 + k; u = (int)(t - k * sl); return; }
    t -= 3 * sl;
    const long long G = 2 * d.pay_len;
    if (G == 0 || t >= ns[G]) { b = d.total_bits; u = 0; return; }
    long long lo = 0, hi = G;                                // last codeword starting at or before t
    while (hi - lo > 1) {
        const long long mid = (lo + hi) >> 1;
        if (ns[mid] <= t) lo = mid; else hi = mid;
    }
    long long rem = t - ns[lo];
    const uint32_t byte = pay[d.pay_off + (lo >> 1)];
    const uint32_t cw = hamming74_encode((lo & 1) ? (byte & 15u) : (byte >> 4));
    int r = 0;
    for (; r < 6; r++) {
        const long long L = ((cw >> r) & 1u) ? ml : sl;
        if (rem < L) break;
        rem -= L;
    }
    b = d.ts_bits + 4 + 7 * lo + r;
    u = (int)rem;
}

// Unequal tones: a lane synthesizes 64 consecutive frames (8 output vectors) into a per-warp staging block in shared
// memory (XOR-swizzled: conflict-free both ways); the warp then writes its 256 vectors as coalesced 128-bit stores.
//
// Tones of at least 8 frames (4800 baud and below): one var_locate, then the lane lists the nine bits its 64 frames can
// touch — symbol and first frame relative to the lane's — in its column of a shared-memory table (inside the coded
// bits the symbols are cut out of one 21-bit stream built from the two payload bytes that hold the three codewords
// involved) and emits its 32 frame pairs WITHOUT A BRANCH: per pair one table load, "has the next bit started" as a
// select, the tone phase as a bit of the tone's mask.  ncu on the walk it replaces (a while loop per pair that
// advanced bit by bit): 14 of 32 lanes active per instruction, 1.04 G warp instructions for 637 M frames, a third of the
// stall samples waiting for instruction fetch — it ran at 0.85 TB/s whatever was done to its searches and its arithmetic.
//
// Shorter tones (8000 baud: 4 / 6 frames; 24000 baud: the mark tone has no frames at all, :81-85) keep that walk: a bit
// list per 64 frames would not be bounded.
constexpr int kVarVecPerLane = 8;
constexpr int kVarBlockVecs = 32 * kVarVecPerLane;           // 256 vectors = 2048 frames per warp step
constexpr int kVarBits = 10;                                 // nine bits per lane step and a sentinel

__global__ void __launch_bounds__(kSynthThreads) k_synth_var(const uint8_t *__restrict__ pay,
                                                             const TxDesc *__restrict__ descs,
                                                             const int32_t *__restrict__ chunk_cap,
                                                             const int64_t *__restrict__ nib_start,
                                                             int16_t *__restrict__ out)
{
    __shared__ uint4 stage[kSynthThreads / 32][kVarBlockVecs];
    __shared__ int32_t bits[kVarBits][kSynthThreads];        // [bit][thread]: (first frame relative to the lane's) * 4 + symbol
    const long long chunk = blockIdx.x;
    const TxDesc d = descs[chunk_cap[chunk]];
    if (d.ml == d.bf) return;                                // equal tones: k_synth
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t *ns = nib_start + d.nib_off;
    const long long nvec_cap = (d.out_len + 7) >> 3;
    const long long v0 = (chunk - d.chunk_first) * kChunkVecs;
    const long long vend = min(v0 + (long long)kChunkVecs, nvec_cap);
    uint4 *dst = reinterpret_cast<uint4 *>(out + d.out_off);
    uint4 *st = stage[warp];
    const bool long_tones = d.ml >= 8;                       // uniform over the CTA
    // tones of up to 64 frames as bit masks over their even phases (bit k: frame 2k is HI; tone_pair's rule, Waveforms :68-85):
    // space = h HI, h LO (h = bf / 2); mark = q HI, q LO, q HI, q LO (q = int(bf / 4))
    const bool use_masks = d.bf <= 64;
    uint32_t mask_mark = 0u, mask_space = 0u;
    if (use_masks) {
        const int q = d.bf >> 2, h = d.bf >> 1;
        auto below = [](int n) -> uint32_t { return n >= 32 ? 0xFFFFFFFFu : ((1u << n) - 1u); };   // bits k with k < n
        mask_space = below((h + 1) >> 1);                                                // 2k < h
        mask_mark = below((q + 1) >> 1) | (below((3 * q + 1) >> 1) & ~below(q));          // 2k < q  or  2q <= 2k < 3q
    }
    const long long first_coded = d.ts_bits + 4;
    for (long long vb = v0 + (long long)warp * kVarBlockVecs; vb < vend; vb += (long long)(kSynthThreads / 32) * kVarBlockVecs) {
        const long long vl = vb + (long long)lane * kVarVecPerLane;      // this lane's first vector
        if (vl < vend && long_tones) {
            long long b;
            int u;
            var_locate(8 * vl, d, pay, ns, b, u);
            // ---- the nine bits from b: symbols
            uint32_t symbits = 0u;                           // two bits per symbol (2 = the zero frames behind the last bit)
            if (b >= first_coded && b + 8 < d.total_bits) {
                const long long j = b - first_coded;         // coded bit index: codeword g0, place r0
                const long long g0 = j < 0x7FFFFFFFLL ? (long long)((uint32_t)j / 7u) : j / 7;   // 32-bit divide for all but > 150 MB payloads
                const int r0 = (int)(j - 7 * g0);
                const long long i0 = g0 >> 1;
                const uint32_t B0 = pay[d.pay_off + i0];
                const uint32_t B1 = (i0 + 1 < d.pay_len) ? pay[d.pay_off + i0 + 1] : 0u;
                const uint32_t B01 = (B0 << 8) | B1;
                uint32_t stream = 0u;
#pragma unroll
                for (int k = 0; k < 3; k++) {
                    const int idx = (int)(g0 & 1) + k;       // nibble 0..3 of the two bytes, high nibble first :446-450
                    stream |= hamming74_encode((B01 >> (12 - 4 * idx)) & 15u) << (7 * k);
                }
                stream >>= r0;
#pragma unroll
                for (int i = 0; i < 9; i++) symbits |= ((stream >> i) & 1u) << (2 * i);
            } else {
#pragma unroll 1
                for (int i = 0; i < 9; i++) symbits |= (b + i < d.total_bits ? tx_bit(b + i, d, pay) : 2u) << (2 * i);
            }
            // ---- first frames relative to the lane's first frame; bit 0 started u frames before it
            int rel = -u;
#pragma unroll
            for (int i = 0; i < 9; i++) {
                const uint32_t sy = (symbits >> (2 * i)) & 3u;
                bits[i][tid] = rel * 4 + (int)sy;
                rel += sy == 2u ? (1 << 20) : (sy ? d.ml : d.bf);
            }
            bits[9][tid] = (1 << 23) + 2;                    // never starts
            // ---- 32 frame pairs: at most one bit starts between two of them (tones of 8 frames and more)
            int cur = 0;
            int curk = bits[0][tid];
#pragma unroll
            for (int k = 0; k < kVarVecPerLane; k++) {
                uint32_t w[4];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const int o = 8 * k + 2 * j;
                    const int nextk = bits[cur + 1][tid];
                    const bool adv = o >= (nextk >> 2);
                    cur += adv ? 1 : 0;
                    curk = adv ? nextk : curk;
                    const uint32_t sy = (uint32_t)curk & 3u;
                    const int ph = o - (curk >> 2);
                    if (use_masks)
                        w[j] = sy == 2u ? 0u : ((((sy ? mask_mark : mask_space) >> ((ph >> 1) & 31)) & 1u) ? 0x7FFF7FFFu : 0x80008000u);
                    else
                        w[j] = tone_pair(sy, ph, d.bf);
                }
                const int v = lane * kVarVecPerLane + k;
                st[v ^ ((v >> 3) & 7)] = make_uint4(w[0], w[1], w[2], w[3]);
            }
        } else if (vl < vend) {
            long long b;
            int u;
            var_locate(8 * vl, d, pay, ns, b, u);
            uint32_t sym = b < d.total_bits ? tx_bit(b, d, pay) : 2u;
            int L = sym == 2u ? 0x7FFFFFFF : (sym ? d.ml : d.bf);
#pragma unroll
            for (int k = 0; k < kVarVecPerLane; k++) {
                uint32_t w[4];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    w[j] = tone_pair(sym, u, d.bf);
                    u += 2;
                    while (u >= L) {                         // next bit of the sequence (__getFrames :463-467 appends tone after tone;
                        u -= L;                              //  at 24000 baud the mark tone has no frames at all, :81-85)
                        b++;
                        sym = b < d.total_bits ? tx_bit(b, d, pay) : 2u;
                        L = sym == 2u ? 0x7FFFFFFF : (sym ? d.ml : d.bf);
                    }
                }
                const int v = lane * kVarVecPerLane + k;
                st[v ^ ((v >> 3) & 7)] = make_uint4(w[0], w[1], w[2], w[3]);
            }
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < kVarVecPerLane; r++) {
            const int v = 32 * r + lane;
            if (vb + v < vend) dst[vb + v] = st[v ^ ((v >> 3) & 7)];
        }
        __syncwarp();
    }
}

static size_t synth_smem_bytes(int bf)
{
    const int G = (bf & 7) ? 2 : 1, VG = G * bf / 8;
    return (size_t)(G == 1 ? 3 : 9) * VG * 16 + kMaxSymbols;
}

// ------------------------------------------------------------------ streaming transmitter ----
// S channels on one shared timeline; channel s's frames [start, start + out_len) of a queued message are
// that message's save() frames, every other frame is 0.  k_tx_window synthesizes the window [P, P + n) of
// every channel straight from payload bytes, as the flat row-major S x n output (row s = channel s).  Its
// descriptors are the TxDescs of the messages that overlap the window, with out_off = the message's first
// frame on the timeline, listed per row (CSR row_off[S + 1]).
//
// Every frame of a message is the even frame of its pair (SoundOutput.__convertFrames :239-244, counted from
// the message's own first frame).  All tone lengths are even (0 included: the 24000-baud mark), so a pair never
// straddles two bits and a frame's value is the tone at its bit phase rounded down to even.
constexpr int kWinThreads = 256;

// bit b and phase u (frames into the bit's tone) of even message frame p: one divide (32-bit below 2^31
// frames) for equal tones, var_locate for unequal ones
__device__ __forceinline__ void win_locate(long long p, const TxDesc &d, const uint8_t *__restrict__ pay,
                                           const int64_t *__restrict__ nib, long long &b, int &u)
{
    if (d.ml != d.bf) { var_locate(p, d, pay, nib + d.nib_off, b, u); return; }
    if (p < 0x7FFFFFFFLL) {
        const uint32_t q = (uint32_t)p / (uint32_t)d.bf;
        b = q; u = (int)((uint32_t)p - q * (uint32_t)d.bf);
    } else {
        b = p / d.bf; u = (int)(p - b * d.bf);
    }
}

__device__ __forceinline__ void win_bit(long long b, const TxDesc &d, const uint8_t *__restrict__ pay, uint32_t &sym, int &L)
{
    sym = b < d.total_bits ? tx_bit(b, d, pay) : 2u;           // 4800 zero frames :468
    L = sym == 2u ? 0x7FFFFFFF : (sym ? d.ml : d.bf);
}

// the window message of row `row` that holds or follows timeline frame t (first with end > t); hi if none
__device__ __forceinline__ int win_find(const TxDesc *__restrict__ descs, int lo, int hi, long long t)
{
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (descs[mid].out_off + descs[mid].out_len <= t) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// one frame of row `row` at timeline frame t (boundary vectors only)
__device__ int16_t win_frame(const TxDesc *__restrict__ descs, const int32_t *__restrict__ row_off, long long row,
                             long long t, const uint8_t *__restrict__ pay, const int64_t *__restrict__ nib)
{
    const int hi = row_off[row + 1];
    const int k = win_find(descs, row_off[row], hi, t);
    if (k >= hi || descs[k].out_off > t) return 0;
    const TxDesc d = descs[k];
    long long b;
    int u;
    win_locate((t - d.out_off) & ~1LL, d, pay, nib, b, u);
    uint32_t sym;
    int L;
    win_bit(b, d, pay, sym, L);
    return (int16_t)(tone_pair(sym, u, d.bf) & 0xFFFFu);
}

// Frames t0 .. t0 + 7 of row `row` (all inside the window row) as one 16-byte vector, into o; false when they
// straddle a message boundary (the caller then computes them frame by frame with win_frame).  A vector inside one
// message locates its first pair once and walks five pairs (the short-tone walk of k_synth_var: at 24000 baud a
// mark has no frames); its words are the pair values, shifted by one frame when the message starts on an odd frame
// of the vector.  Silence is zero.
__device__ __forceinline__ bool win_vec(const TxDesc *__restrict__ descs, const int32_t *__restrict__ row_off, long long row,
                                        long long t0, const uint8_t *__restrict__ pay, const int64_t *__restrict__ nib, uint4 &o)
{
    const int hi = row_off[row + 1];
    const int k = win_find(descs, row_off[row], hi, t0);
    if (k >= hi || descs[k].out_off >= t0 + 8) {               // silence
        o = make_uint4(0u, 0u, 0u, 0u);
        return true;
    }
    const TxDesc d = descs[k];
    if (d.out_off > t0 || d.out_off + d.out_len < t0 + 8) return false;
    const long long m0 = t0 - d.out_off;
    long long b;
    int u;
    win_locate(m0 & ~1LL, d, pay, nib, b, u);
    uint32_t sym;
    int L;
    win_bit(b, d, pay, sym, L);
    uint32_t pv[5];
#pragma unroll
    for (int j = 0; j < 5; j++) {
        pv[j] = tone_pair(sym, u, d.bf);
        u += 2;
        while (u >= L) {                                       // next bit (__getFrames :463-467 appends tone after tone)
            u -= L;
            b++;
            win_bit(b, d, pay, sym, L);
        }
    }
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; j++) w[j] = (m0 & 1) ? ((pv[j] & 0xFFFFu) | (pv[j + 1] & 0xFFFF0000u)) : pv[j];
    o = make_uint4(w[0], w[1], w[2], w[3]);
    return true;
}

// The planar window, out[s * n + c] = frame P + c of channel s: one thread per 16-byte output vector.  A vector
// inside one row is win_vec's; one across a row or message boundary, or at the end of the output, writes its frames
// one by one.
__global__ void __launch_bounds__(kWinThreads) k_tx_window(const uint8_t *__restrict__ pay, const int64_t *__restrict__ nib,
                                                           const TxDesc *__restrict__ descs, const int32_t *__restrict__ row_off,
                                                           long long P, long long n, long long total, int16_t *__restrict__ out)
{
    const long long v = (long long)blockIdx.x * kWinThreads + threadIdx.x;
    const long long f0 = 8 * v;
    if (f0 >= total) return;
    long long row, col;
    if (f0 < 0xFFFFFFFFLL && n < 0xFFFFFFFFLL) {
        const uint32_t r32 = (uint32_t)f0 / (uint32_t)n;
        row = r32; col = f0 - (long long)r32 * n;
    } else {
        row = f0 / n; col = f0 - row * n;
    }
    uint4 o;
    if (col + 8 <= n && win_vec(descs, row_off, row, P + col, pay, nib, o)) {
        *reinterpret_cast<uint4 *>(out + f0) = o;
        return;
    }
#pragma unroll 1
    for (int e = 0; e < 8 && f0 + e < total; e++) {
        out[f0 + e] = win_frame(descs, row_off, row, P + col, pay, nib);
        if (++col == n) { col = 0; row++; }
    }
}

// k_tx_window_frames<Tout>: the interleaved window, written into a window of a wider output: frame P + c of channel s,
// converted by the rule of the output format (sample_from_s16), is element e0 + c * pitch + s of out (out 16-byte
// aligned, e0 < 16 / sizeof(Tout) the window's offset in its first vector, pitch >= S): what a multi-channel sound card
// takes, or some columns of it. A CTA computes kIlC consecutive channels x kIlV column vectors of 8 frames (aligned on
// the window column, so no vector straddles two channels) with win_vec, or win_frame for a vector across a message
// boundary or the window's end: one thread per vector, consecutive threads along a channel as in k_tx_window, into
// shared memory. It then writes the tile frame-major: each of its frame rows is the contiguous run of kIlC samples at
// e0 + f * pitch + c0, written from its absolute alignment as aligned 16-byte vectors of the output, the row's partial
// head and tail vectors sample by sample, so nothing outside the window is written and handles may fill disjoint
// windows of one buffer. Shared rows are channels in the order (s & 7) * 8 + (s >> 3), 136 samples apart, so that the
// lanes of one output row read consecutive shared rows in distinct bank groups.
constexpr int kIlC = 64, kIlV = 16, kIlStride = 8 * kIlV + 8;

// k_tx_window_frames<int16_t> for a contiguous, 16-byte aligned output (pitch S, e0 = 0), the layout of
// afsk_tx_streams_pull_interleaved: its row arithmetic is cheaper, and it measured faster (DESIGN.md §5)
__global__ void __launch_bounds__(kWinThreads) k_tx_window_interleaved(const uint8_t *__restrict__ pay, const int64_t *__restrict__ nib,
                                                                       const TxDesc *__restrict__ descs,
                                                                       const int32_t *__restrict__ row_off, long long P, long long n,
                                                                       int S, int cblocks, int16_t *__restrict__ out)
{
    __shared__ __align__(16) int16_t T[kIlC * kIlStride];
    const int c0 = (int)(blockIdx.x % cblocks) * kIlC, nc = min(kIlC, S - c0);
    const long long F0 = (long long)(blockIdx.x / cblocks) * (8 * kIlV);
    const int nf = (int)min(8LL * kIlV, n - F0);
    const int col = 8 * (threadIdx.x % kIlV);                    // this thread's column vector, on every channel
    if (col < nf) {
        const long long t0 = P + F0 + col;
        const int m = min(8, nf - col);
#pragma unroll 1
        for (int c = threadIdx.x / kIlV; c < nc; c += kWinThreads / kIlV) {
            uint4 o;
            if (m < 8 || !win_vec(descs, row_off, c0 + c, t0, pay, nib, o)) {   // frame by frame, 0 past the window
                unsigned long long w = 0, x = 0;
#pragma unroll 1
                for (int e = 0; e < m; e++) {
                    const unsigned long long f = (uint16_t)win_frame(descs, row_off, c0 + c, t0 + e, pay, nib);
                    if (e < 4) w |= f << (16 * e); else x |= f << (16 * (e - 4));
                }
                o = make_uint4((uint32_t)w, (uint32_t)(w >> 32), (uint32_t)x, (uint32_t)(x >> 32));
            }
            *reinterpret_cast<uint4 *>(T + ((c & 7) * 8 + (c >> 3)) * kIlStride + col) = o;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nf * 9; i += kWinThreads) {     // a row of kIlC samples spans at most 9 vectors
        const int q = i % 9, fl = i / 9;
        const long long a = (F0 + fl) * S + c0, b = a + nc;      // the row's samples in out
        const long long d0 = ((a >> 3) + q) * 8;
        if (d0 >= b) continue;
        uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int e = 0; e < 8; e++) {
            const int c = (int)(d0 + e - a);
            if (c >= 0 && c < nc) w[e >> 1] |= (uint32_t)(uint16_t)T[((c & 7) * 8 + (c >> 3)) * kIlStride + fl] << (16 * (e & 1));
        }
        if (d0 >= a && d0 + 8 <= b) {
            *reinterpret_cast<uint4 *>(out + d0) = make_uint4(w[0], w[1], w[2], w[3]);
        } else {
#pragma unroll
            for (int e = 0; e < 8; e++)
                if (d0 + e >= a && d0 + e < b) out[d0 + e] = (int16_t)(w[e >> 1] >> (16 * (e & 1)));
        }
    }
}

// (__maxnreg__ in place of __launch_bounds__(kWinThreads): with the calls of the synthesis loop, ptxas otherwise settles
// on 40 registers and spills two values across them)
template <typename Tout>
__global__ void __maxnreg__(48) k_tx_window_frames(const uint8_t *__restrict__ pay, const int64_t *__restrict__ nib,
                                                                       const TxDesc *__restrict__ descs,
                                                                       const int32_t *__restrict__ row_off, long long P, long long n,
                                                                       int S, int cblocks, long long pitch, int e0,
                                                                       Tout *__restrict__ out)
{
    constexpr int V = 16 / sizeof(Tout), NV = kIlC / V + 1;      // samples per vector; a row spans at most NV vectors
    __shared__ __align__(16) int16_t T[kIlC * kIlStride];
    const int c0 = (int)(blockIdx.x % cblocks) * kIlC, nc = min(kIlC, S - c0);
    const long long F0 = (long long)(blockIdx.x / cblocks) * (8 * kIlV);
    const int nf = (int)min(8LL * kIlV, n - F0);
    const int col = 8 * (threadIdx.x % kIlV);                    // this thread's column vector, on every channel
    if (col < nf) {
        const long long t0 = P + F0 + col;
        const int m = min(8, nf - col);
#pragma unroll 1
        for (int c = threadIdx.x / kIlV; c < nc; c += kWinThreads / kIlV) {
            uint4 o;
            if (m < 8 || !win_vec(descs, row_off, c0 + c, t0, pay, nib, o)) {   // frame by frame, 0 past the window
                unsigned long long w = 0, x = 0;
#pragma unroll 1
                for (int e = 0; e < m; e++) {
                    const unsigned long long f = (uint16_t)win_frame(descs, row_off, c0 + c, t0 + e, pay, nib);
                    if (e < 4) w |= f << (16 * e); else x |= f << (16 * (e - 4));
                }
                o = make_uint4((uint32_t)w, (uint32_t)(w >> 32), (uint32_t)x, (uint32_t)(x >> 32));
            }
            *reinterpret_cast<uint4 *>(T + ((c & 7) * 8 + (c >> 3)) * kIlStride + col) = o;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nf * NV; i += kWinThreads) {
        const int q = i % NV, fl = i / NV;
        const long long a = e0 + (F0 + fl) * pitch + c0, b = a + nc;    // the row's samples in out
        const long long d0 = ((a >> (V == 8 ? 3 : 2)) + q) * V;
        if (d0 >= b) continue;
        Tout w[V];
#pragma unroll
        for (int e = 0; e < V; e++) {
            const int c = (int)(d0 + e - a);
            w[e] = c >= 0 && c < nc ? sample_from_s16<Tout>(T[((c & 7) * 8 + (c >> 3)) * kIlStride + fl]) : Tout(0);
        }
        if (d0 >= a && d0 + V <= b) {
            uint4 v;
            memcpy(&v, w, 16);
            *reinterpret_cast<uint4 *>(out + d0) = v;
        } else {
#pragma unroll
            for (int e = 0; e < V; e++)
                if (d0 + e >= a && d0 + e < b) out[d0 + e] = w[e];
        }
    }
}

// Moves live arena blocks (16-byte aligned, whole 16-byte units) into the other arena: one CTA per block.
struct TxMove { long long src, dst, len; };

__global__ void __launch_bounds__(kWinThreads) k_tx_compact(const uint4 *__restrict__ src, uint4 *__restrict__ dst,
                                                            const TxMove *__restrict__ mv)
{
    const TxMove m = mv[blockIdx.x];
    for (long long i = threadIdx.x; i < m.len / 16; i += kWinThreads) dst[m.dst / 16 + i] = src[m.src / 16 + i];
}

}  // namespace

struct AfskTxPlan {
    int device = 0;
    int B = 0;
    std::vector<TxDesc> descs;
    std::vector<int64_t> out_off, out_len;
    TxDesc *d_descs = nullptr;
    int32_t *d_chunk_cap = nullptr;
    std::vector<int32_t> chunk_cap;
    int64_t total_chunks = 0;
    size_t smem = 0;
    std::vector<int32_t> var_caps;       // captures with unequal mark/space tone lengths
    int32_t *d_var_caps = nullptr;
    int64_t *d_nib_start = nullptr;
    int64_t nib_entries = 0;
    bool has_equal = false;
};

extern "C" {

int64_t afsk_tx_num_samples(int baud, int64_t ts_cycles, int64_t payload_bytes, const uint8_t *payload)
{
    int bf, ml, sl;
    if (!afsk_tone_geometry(baud, &bf, &ml, &sl)) { afsk_set_error("Invalid baud rate."); return AFSK_E_BAUD; }
    if (ts_cycles < 0) ts_cycles = 0;
    int64_t frames = ts_cycles * (int64_t)(ml + sl) + ml + 3 * (int64_t)sl + AFSK_TAIL_FRAMES;
    if (ml == sl) {
        frames += payload_bytes * 14 * (int64_t)sl;
    } else {
        if (payload_bytes > 0 && !payload) { afsk_set_error("payload needed for unequal tone lengths"); return AFSK_E_ARG; }
        for (int64_t i = 0; i < payload_bytes; i++) {
            for (int half = 0; half < 2; half++) {
                uint32_t v = half == 0 ? payload[i] >> 4 : payload[i] & 15u;
                uint32_t d0 = (v >> 3) & 1u, d1 = (v >> 2) & 1u, d2 = (v >> 1) & 1u, d3 = v & 1u;
                int ones = (int)((d0 ^ d1 ^ d3) + (d0 ^ d2 ^ d3) + d0 + (d1 ^ d2 ^ d3) + d1 + d2 + d3);
                frames += (int64_t)ones * ml + (int64_t)(7 - ones) * sl;
            }
        }
    }
    return frames & ~(int64_t)1;      // SoundOutput.__convertFrames :241 drops an odd trailing frame
}

int afsk_tx_plan_create(int device, int B, const int64_t *h_pay_off, const int32_t *h_baud, const int64_t *h_ts_cycles,
                        const uint8_t *h_payload, AfskTxPlan **plan_out)
{
    if (!plan_out || B < 0 || (B > 0 && (!h_pay_off || !h_baud || !h_ts_cycles))) return AFSK_E_ARG;
    AfskDeviceGuard guard(device);
    if (!guard.ok) { afsk_set_error("cannot select device %d", device); return AFSK_E_CUDA; }
    AfskTxPlan *P = new (std::nothrow) AfskTxPlan();
    if (!P) return AFSK_E_ARG;
    P->device = device;
    P->B = B;
    P->descs.resize(B);
    P->out_off.assign(B + 1, 0);
    P->out_len.assign(B, 0);
    int64_t chunks = 0;
    for (int c = 0; c < B; c++) {
        int bf, ml, sl;
        if (!afsk_tone_geometry(h_baud[c], &bf, &ml, &sl)) {
            delete P; afsk_set_error("Invalid baud rate."); return AFSK_E_BAUD;
        }
        TxDesc &d = P->descs[c];
        const int64_t ts = h_ts_cycles[c] < 0 ? 0 : h_ts_cycles[c];
        d.pay_off = h_pay_off[c];
        d.pay_len = h_pay_off[c + 1] - h_pay_off[c];
        if (d.pay_len < 0) { delete P; afsk_set_error("payload offsets must be non-decreasing"); return AFSK_E_ARG; }
        d.bf = bf; d.ml = ml; d.pad = 0; d.nib_off = 0;
        d.ts_bits = 2 * ts;
        d.total_bits = d.ts_bits + 4 + 14 * d.pay_len;
        if (ml == sl) {
            d.out_len = (d.total_bits * bf + AFSK_TAIL_FRAMES) & ~(int64_t)1;
            P->smem = std::max(P->smem, synth_smem_bytes(bf));
            P->has_equal = true;
        } else {
            // the length depends on how many mark bits the codewords hold: the plan is made for THIS payload
            if (d.pay_len > 0 && !h_payload) {
                delete P; afsk_set_error("afsk_tx_plan_create: the payload is needed for baud %d (unequal tone lengths)", h_baud[c]);
                return AFSK_E_ARG;
            }
            const int64_t nf = afsk_tx_num_samples(h_baud[c], ts, d.pay_len, h_payload ? h_payload + d.pay_off : nullptr);
            if (nf < 0) { delete P; return (int)nf; }
            d.out_len = nf;
            d.nib_off = P->nib_entries;
            P->nib_entries += 2 * d.pay_len + 1;
            P->var_caps.push_back(c);
        }
        d.out_off = P->out_off[c];
        d.chunk_first = chunks;
        const int64_t nvec = (d.out_len + 7) >> 3;
        const int64_t nch = (nvec + kChunkVecs - 1) / kChunkVecs;
        if (chunks + nch > 0x7FFFFFF0LL) { delete P; afsk_set_error("batch too large"); return AFSK_E_ARG; }
        P->chunk_cap.insert(P->chunk_cap.end(), (size_t)nch, (int32_t)c);
        chunks += nch;
        P->out_len[c] = d.out_len;
        P->out_off[c + 1] = P->out_off[c] + nvec * 8;
    }
    P->total_chunks = chunks;
    if (chunks > 0x7FFFFFFFLL) { delete P; afsk_set_error("batch too large"); return AFSK_E_ARG; }
    if (P->smem > 200 * 1024) { delete P; afsk_set_error("bit_frames too large for the synthesizer"); return AFSK_E_UNSUPPORTED; }
    cudaError_t e = cudaMalloc((void **)&P->d_descs, sizeof(TxDesc) * (B ? B : 1));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_synth, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e == cudaSuccess && B) e = cudaMemcpy(P->d_descs, P->descs.data(), sizeof(TxDesc) * B, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc((void **)&P->d_chunk_cap, sizeof(int32_t) * (chunks ? chunks : 1));
    if (e == cudaSuccess && chunks)
        e = cudaMemcpy(P->d_chunk_cap, P->chunk_cap.data(), sizeof(int32_t) * chunks, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && !P->var_caps.empty()) {
        e = cudaMalloc((void **)&P->d_var_caps, sizeof(int32_t) * P->var_caps.size());
        if (e == cudaSuccess) e = cudaMemcpy(P->d_var_caps, P->var_caps.data(), sizeof(int32_t) * P->var_caps.size(), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMalloc((void **)&P->d_nib_start, sizeof(int64_t) * P->nib_entries);
    }
    if (e != cudaSuccess) {
        afsk_set_error("afsk_tx_plan_create: %s", cudaGetErrorString(e));
        afsk_tx_plan_destroy(P);
        return AFSK_E_CUDA;
    }
    *plan_out = P;
    return AFSK_OK;
}

int afsk_tx_plan_destroy(AfskTxPlan *P)
{
    if (!P) return AFSK_OK;
    AfskDeviceGuard guard(P->device);
    cudaFree(P->d_descs);
    cudaFree(P->d_chunk_cap);
    cudaFree(P->d_var_caps);
    cudaFree(P->d_nib_start);
    delete P;
    return AFSK_OK;
}

int afsk_tx_plan_out_offsets(const AfskTxPlan *P, const int64_t **h_out_off, const int64_t **h_out_len)
{
    if (!P) return AFSK_E_ARG;
    if (h_out_off) *h_out_off = P->out_off.data();
    if (h_out_len) *h_out_len = P->out_len.data();
    return AFSK_OK;
}

int afsk_tx_synth(AfskTxPlan *P, const uint8_t *d_payload, int16_t *d_out, void *stream)
{
    if (!P || (P->B > 0 && !d_out)) return AFSK_E_ARG;
    if ((reinterpret_cast<uintptr_t>(d_out) & 15) != 0) { afsk_set_error("afsk_tx_synth: d_out must be 16-byte aligned"); return AFSK_E_ARG; }
    if (P->B == 0 || P->total_chunks == 0) return AFSK_OK;
    AfskDeviceGuard guard(P->device);
    if (!guard.ok) return AFSK_E_CUDA;
    cudaStream_t st = (cudaStream_t)stream;
    if (P->has_equal)
        k_synth<<<(unsigned)P->total_chunks, kSynthThreads, P->smem, st>>>(d_payload, P->d_descs, P->d_chunk_cap, d_out);
    if (!P->var_caps.empty()) {
        k_tx_nibscan<<<(unsigned)P->var_caps.size(), kScanThreads, 0, st>>>(d_payload, P->d_descs, P->d_var_caps, P->d_nib_start);
        k_synth_var<<<(unsigned)P->total_chunks, kSynthThreads, 0, st>>>(d_payload, P->d_descs, P->d_chunk_cap, P->d_nib_start, d_out);
    }
    AFSK_CUDA(cudaGetLastError());
    return AFSK_OK;
}

int afsk_tx_synth_host(int device, const uint8_t *h_payload, const int64_t *h_pay_off, int B, const int32_t *h_baud,
                       const int64_t *h_ts_cycles, int16_t *h_out, const int64_t *h_out_off)
{
    if (B < 0 || (B > 0 && (!h_pay_off || !h_out || !h_out_off))) return AFSK_E_ARG;
    if (B == 0) return AFSK_OK;
    AfskTxPlan *P = nullptr;
    int rc = afsk_tx_plan_create(device, B, h_pay_off, h_baud, h_ts_cycles, h_payload, &P);
    if (rc) return rc;
    AfskDeviceGuard guard(device);
    const int64_t pay_bytes = h_pay_off[B];
    uint8_t *d_pay = nullptr; int16_t *d_out = nullptr;
    cudaError_t e = cudaMalloc((void **)&d_pay, (size_t)(pay_bytes ? pay_bytes : 16));
    if (e == cudaSuccess) e = cudaMalloc((void **)&d_out, (size_t)(P->out_off[B] ? P->out_off[B] : 8) * 2);
    if (e == cudaSuccess && pay_bytes) e = cudaMemcpy(d_pay, h_payload, (size_t)pay_bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        rc = afsk_tx_synth(P, d_pay, d_out, nullptr);
        for (int c = 0; c < B && rc == AFSK_OK && e == cudaSuccess; c++) {
            if (h_out_off[c + 1] - h_out_off[c] < P->out_len[c]) { rc = AFSK_E_ARG; afsk_set_error("output capacity too small for capture %d", c); break; }
            if (P->out_len[c])
                e = cudaMemcpy(h_out + h_out_off[c], d_out + P->out_off[c], (size_t)P->out_len[c] * 2, cudaMemcpyDeviceToHost);
        }
    }
    cudaFree(d_pay); cudaFree(d_out);
    afsk_tx_plan_destroy(P);
    if (e != cudaSuccess) { afsk_set_error("afsk_tx_synth_host: %s", cudaGetErrorString(e)); return AFSK_E_CUDA; }
    return rc;
}

}  // extern "C"

// ---------------------------------------------------------------- streaming transmitter (host) ----
// Device state is O(payload bytes): one arena of 16-byte aligned blocks, one per queued message: its payload
// and, for unequal tones, its codeword start table (k_tx_nibscan at send time).  New blocks go on top.  When
// they do not fit, the live blocks move (k_tx_compact) to the bottom of the other arena, whose capacity doubles
// until the live blocks and the new ones fill at most half of it.  A compaction therefore follows at least half
// an arena of sent bytes and moves at most one arena: moved bytes per sent byte stay below 2.  A message is
// retired once the timeline has passed its end; when none is left, the top returns to the bottom.
namespace {
constexpr int64_t kTxArenaMin = 65536;
int64_t round16(int64_t x) { return (x + 15) & ~(int64_t)15; }

struct TxMsg {
    int64_t block_off, block_bytes;
    TxDesc d;                       // pay_off / nib_off into the arena, out_off = first frame on the timeline
};
}  // namespace

struct AfskTxStreams {
    int device = 0, S = 0;
    // per channel: the settings of the messages it is sent next (bf, ml: tone lengths of baud)
    std::vector<int32_t> baud, bf, ml;
    std::vector<int64_t> ts_cycles;
    int64_t P = 0;                                        // frames pulled
    std::vector<std::deque<TxMsg>> q;                     // per channel: messages not yet fully pulled
    std::vector<int64_t> last_end;                        // per channel: end of the last message sent
    uint8_t *arena[2] = {nullptr, nullptr};
    size_t arena_alloc[2] = {0, 0};
    int cur = 0;
    int64_t cap = 0, top = 0, live = 0;                   // bytes: capacity of the current arena, used, in live blocks
    bool failed = false;
    int64_t n_launches = 0, n_moved = 0, n_compactions = 0;
    uint8_t *h_stage = nullptr; size_t h_stage_cap = 0;   // pinned: new blocks / descriptors of one call
    uint8_t *d_scratch = nullptr; size_t d_scratch_cap = 0;
    int16_t *d_out = nullptr; size_t out_cap = 0;         // pull into host memory
};

// a send or pull with valid arguments: any failure may leave the queues and the arena between two states, so the
// handle refuses every later send / pull
template <typename F> static int tx_streams_call(AfskTxStreams *H, F run)
{
    if (H->failed) { afsk_set_error("afsk_tx_streams: an earlier call failed; destroy the handle"); return AFSK_E_CUDA; }
    AfskDeviceGuard guard(H->device);
    if (!guard.ok) { afsk_set_error("cannot select device %d", H->device); return AFSK_E_CUDA; }
    const int rc = run();
    if (rc != AFSK_OK) H->failed = true;
    return rc;
}

// a send with valid arguments: synchronous on the legacy default stream
static int tx_send_run(AfskTxStreams *H, int n, const int32_t *h_stream, const int64_t *h_pay_off, const uint8_t *h_payload,
                       int64_t *h_start, int64_t *h_end)
{
    if (n == 0) return AFSK_OK;
    cudaStream_t st = nullptr;

    // the new blocks, in order, above the top (after a compaction if they do not fit), each with its channel's
    // settings; var: the messages with unequal tone lengths, whose blocks also hold a codeword start table
    std::vector<TxMsg> msgs((size_t)n);
    std::vector<int32_t> var;
    int64_t W = 0;
    for (int i = 0; i < n; i++) {
        const int s = h_stream[i];
        TxMsg &m = msgs[i];
        TxDesc &d = m.d;
        memset(&d, 0, sizeof(d));
        d.pay_len = h_pay_off[i + 1] - h_pay_off[i];
        d.bf = H->bf[s]; d.ml = H->ml[s];
        d.ts_bits = 2 * H->ts_cycles[s];
        d.total_bits = d.ts_bits + 4 + 14 * d.pay_len;
        d.out_len = afsk_tx_num_samples(H->baud[s], H->ts_cycles[s], d.pay_len, d.pay_len ? h_payload + h_pay_off[i] : nullptr);
        if (d.ml != d.bf) var.push_back(i);
        m.block_off = W;
        m.block_bytes = round16(d.pay_len) + (d.ml != d.bf ? round16(8 * (2 * d.pay_len + 1)) : 0);
        W += m.block_bytes;
    }
    if (H->top + W > H->cap) {
        int64_t newcap = H->cap;
        while (2 * (H->live + W) > newcap) newcap *= 2;
        const int nxt = H->cur ^ 1;
        std::vector<TxMove> mv;
        int64_t o = 0;
        for (auto &qs : H->q)
            for (TxMsg &m : qs) {
                if (m.block_bytes) mv.push_back(TxMove{m.block_off, o, m.block_bytes});
                m.block_off = o;
                m.d.pay_off = o;
                m.d.nib_off = (o + round16(m.d.pay_len)) / 8;
                o += m.block_bytes;
            }
        AFSK_CUDA(grow_device((void **)&H->arena[nxt], &H->arena_alloc[nxt], (size_t)newcap));
        if (!mv.empty()) {
            AFSK_CUDA(grow_pinned((void **)&H->h_stage, &H->h_stage_cap, sizeof(TxMove) * mv.size()));
            AFSK_CUDA(grow_device((void **)&H->d_scratch, &H->d_scratch_cap, sizeof(TxMove) * mv.size()));
            memcpy(H->h_stage, mv.data(), sizeof(TxMove) * mv.size());
            AFSK_CUDA(cudaMemcpyAsync(H->d_scratch, H->h_stage, sizeof(TxMove) * mv.size(), cudaMemcpyHostToDevice, st));
            k_tx_compact<<<(unsigned)mv.size(), kWinThreads, 0, st>>>(reinterpret_cast<const uint4 *>(H->arena[H->cur]),
                                                                     reinterpret_cast<uint4 *>(H->arena[nxt]),
                                                                     reinterpret_cast<const TxMove *>(H->d_scratch));
            AFSK_CUDA(cudaGetLastError());
            AFSK_CUDA(cudaStreamSynchronize(st));    // the scratch and staging are reused below
            H->n_launches++;
        }
        H->n_moved += H->live;
        H->n_compactions++;
        H->cur = nxt;
        H->cap = newcap;
        H->top = H->live;
    }
    // payload image of the new blocks (one copy), then the codeword start tables of unequal-tone messages
    const size_t desc_bytes = var.empty() ? 0 : sizeof(TxDesc) * (size_t)n, caps_bytes = sizeof(int32_t) * var.size();
    AFSK_CUDA(grow_pinned((void **)&H->h_stage, &H->h_stage_cap, (size_t)W + desc_bytes + caps_bytes));
    AFSK_CUDA(grow_device((void **)&H->d_scratch, &H->d_scratch_cap, desc_bytes + caps_bytes + 16));
    for (int i = 0; i < n; i++) {
        TxMsg &m = msgs[i];
        if (m.d.pay_len) memcpy(H->h_stage + m.block_off, h_payload + h_pay_off[i], (size_t)m.d.pay_len);
        m.block_off += H->top;
        m.d.pay_off = m.block_off;
        m.d.nib_off = (m.block_off + round16(m.d.pay_len)) / 8;
    }
    if (W > 0) AFSK_CUDA(cudaMemcpyAsync(H->arena[H->cur] + H->top, H->h_stage, (size_t)W, cudaMemcpyHostToDevice, st));
    if (!var.empty()) {
        TxDesc *hd = reinterpret_cast<TxDesc *>(H->h_stage + W);        // W is a multiple of 16
        int32_t *hc = reinterpret_cast<int32_t *>(H->h_stage + W + desc_bytes);
        for (int i = 0; i < n; i++) hd[i] = msgs[i].d;
        memcpy(hc, var.data(), caps_bytes);
        AFSK_CUDA(cudaMemcpyAsync(H->d_scratch, hd, desc_bytes + caps_bytes, cudaMemcpyHostToDevice, st));
        k_tx_nibscan<<<(unsigned)var.size(), kScanThreads, 0, st>>>(H->arena[H->cur], reinterpret_cast<const TxDesc *>(H->d_scratch),
                                                           reinterpret_cast<const int32_t *>(H->d_scratch + desc_bytes),
                                                           reinterpret_cast<int64_t *>(H->arena[H->cur]));
        AFSK_CUDA(cudaGetLastError());
        H->n_launches++;
    }
    AFSK_CUDA(cudaStreamSynchronize(st));
    H->top += W;
    H->live += W;
    for (int i = 0; i < n; i++) {
        TxMsg &m = msgs[i];
        const int s = h_stream[i];
        m.d.out_off = std::max(H->P, H->last_end[s]);
        H->last_end[s] = m.d.out_off + m.d.out_len;
        h_start[i] = m.d.out_off;
        h_end[i] = H->last_end[s];
        H->q[s].push_back(m);
    }
    return AFSK_OK;
}

// the window as S x n_frames row-major int16 (planar) or interleaved: frame f of channel s at dst[f * pitch + s] in the
// AFSK_SAMPLE_* format (host output: synthesized packed, then copied row by row)
static int tx_pull_run(AfskTxStreams *H, int64_t n_frames, void *dst, int on_device, bool interleaved, int format, int64_t pitch,
                       cudaStream_t st)
{
    if (n_frames == 0) return AFSK_OK;
    const int S = H->S;
    const int64_t n = n_frames, total = (int64_t)S * n, wend = H->P + n;
    const int64_t nvec = (total + 7) >> 3;
    // per row, the messages that overlap [P, P + n): a prefix of the channel's queue (retired ones are gone)
    int64_t nwin = 0;
    for (int s = 0; s < S; s++)
        for (const TxMsg &m : H->q[s]) {
            if (m.d.out_off >= wend) break;
            nwin++;
        }
    const size_t desc_bytes = sizeof(TxDesc) * (size_t)nwin, bytes = desc_bytes + sizeof(int32_t) * ((size_t)S + 1);
    AFSK_CUDA(grow_pinned((void **)&H->h_stage, &H->h_stage_cap, bytes));
    AFSK_CUDA(grow_device((void **)&H->d_scratch, &H->d_scratch_cap, bytes));
    const int size = interleaved ? afsk_sample_size(format) : 2;
    if (!on_device) AFSK_CUDA(grow_device((void **)&H->d_out, &H->out_cap, ((size_t)total * size + 15) / 16 * 16));
    TxDesc *hd = reinterpret_cast<TxDesc *>(H->h_stage);
    int32_t *row_off = reinterpret_cast<int32_t *>(H->h_stage + desc_bytes);
    int32_t k = 0;
    for (int s = 0; s < S; s++) {
        row_off[s] = k;
        for (const TxMsg &m : H->q[s]) {
            if (m.d.out_off >= wend) break;
            hd[k++] = m.d;
        }
    }
    row_off[S] = k;
    AFSK_CUDA(cudaMemcpyAsync(H->d_scratch, H->h_stage, bytes, cudaMemcpyHostToDevice, st));
    // device output is written from the 16-byte vector holding its first sample, e0 samples in
    void *out = on_device ? reinterpret_cast<void *>(reinterpret_cast<uintptr_t>(dst) & ~(uintptr_t)15) : H->d_out;
    const int e0 = on_device ? (int)((reinterpret_cast<uintptr_t>(dst) & 15) / size) : 0;
    const int64_t kpitch = on_device ? pitch : S;
    const uint8_t *a = H->arena[H->cur];
    const int64_t *nib = reinterpret_cast<const int64_t *>(a);
    const TxDesc *d_descs = reinterpret_cast<const TxDesc *>(H->d_scratch);
    const int32_t *d_row_off = reinterpret_cast<const int32_t *>(H->d_scratch + desc_bytes);
    if (interleaved) {
        const int cblocks = (S + kIlC - 1) / kIlC;
        const unsigned grid = (unsigned)(cblocks * ((n + 8 * kIlV - 1) / (8 * kIlV)));
        if (format == AFSK_SAMPLE_S16 && kpitch == S && e0 == 0)
            k_tx_window_interleaved<<<grid, kWinThreads, 0, st>>>(a, nib, d_descs, d_row_off, H->P, n, S, cblocks,
                                                                  static_cast<int16_t *>(out));
        else if (format == AFSK_SAMPLE_S16)
            k_tx_window_frames<<<grid, kWinThreads, 0, st>>>(a, nib, d_descs, d_row_off, H->P, n, S, cblocks, kpitch, e0,
                                                             static_cast<int16_t *>(out));
        else if (format == AFSK_SAMPLE_S32)
            k_tx_window_frames<<<grid, kWinThreads, 0, st>>>(a, nib, d_descs, d_row_off, H->P, n, S, cblocks, kpitch, e0,
                                                             static_cast<int32_t *>(out));
        else
            k_tx_window_frames<<<grid, kWinThreads, 0, st>>>(a, nib, d_descs, d_row_off, H->P, n, S, cblocks, kpitch, e0,
                                                             static_cast<float *>(out));
    } else {
        k_tx_window<<<(unsigned)((nvec + kWinThreads - 1) / kWinThreads), kWinThreads, 0, st>>>(
            a, nib, d_descs, d_row_off, H->P, n, total, static_cast<int16_t *>(out));
    }
    AFSK_CUDA(cudaGetLastError());
    H->n_launches++;
    if (!on_device && interleaved)
        AFSK_CUDA(cudaMemcpy2DAsync(dst, (size_t)pitch * size, H->d_out, (size_t)S * size, (size_t)S * size, (size_t)n,
                                    cudaMemcpyDeviceToHost, st));
    else if (!on_device)
        AFSK_CUDA(cudaMemcpyAsync(dst, H->d_out, (size_t)total * 2, cudaMemcpyDeviceToHost, st));
    AFSK_CUDA(cudaStreamSynchronize(st));
    H->P = wend;
    for (auto &qs : H->q)
        while (!qs.empty() && qs.front().d.out_off + qs.front().d.out_len <= H->P) {
            H->live -= qs.front().block_bytes;
            qs.pop_front();
        }
    if (H->live == 0) H->top = 0;
    return AFSK_OK;
}

extern "C" {

int afsk_tx_streams_create_each(int device, int S, const int32_t *h_baud, const int64_t *h_ts_cycles, AfskTxStreams **h)
{
    if (!h || S < 1 || !h_baud || !h_ts_cycles) {
        afsk_set_error("afsk_tx_streams_create_each: bad argument (S >= 1, non-null arrays)");
        return AFSK_E_ARG;
    }
    int bf, ml, sl;
    for (int s = 0; s < S; s++)
        if (!afsk_tone_geometry(h_baud[s], &bf, &ml, &sl)) {
            afsk_set_error("Invalid baud rate. (afsk_tx_streams_create_each: channel %d, baud %d)", s, h_baud[s]);
            return AFSK_E_BAUD;
        }
    AfskDeviceGuard guard(device);
    if (!guard.ok) { afsk_set_error("cannot select device %d", device); return AFSK_E_CUDA; }
    AfskTxStreams *H = new (std::nothrow) AfskTxStreams();
    if (!H) return AFSK_E_ARG;
    H->device = device; H->S = S;
    H->baud.resize((size_t)S); H->bf.resize((size_t)S); H->ml.resize((size_t)S); H->ts_cycles.resize((size_t)S);
    for (int s = 0; s < S; s++) {
        afsk_tone_geometry(h_baud[s], &bf, &ml, &sl);
        H->baud[s] = h_baud[s]; H->bf[s] = bf; H->ml[s] = ml;
        H->ts_cycles[s] = h_ts_cycles[s] < 0 ? 0 : h_ts_cycles[s];
    }
    H->q.resize((size_t)S);
    H->last_end.assign((size_t)S, 0);
    H->cap = kTxArenaMin;
    const cudaError_t e = grow_device((void **)&H->arena[0], &H->arena_alloc[0], (size_t)H->cap);
    if (e != cudaSuccess) {
        afsk_set_error("afsk_tx_streams_create: %s", cudaGetErrorString(e));
        afsk_tx_streams_destroy(H);
        return AFSK_E_CUDA;
    }
    *h = H;
    return AFSK_OK;
}

int afsk_tx_streams_create(int device, int S, int baud, int64_t ts_cycles, AfskTxStreams **h)
{
    const size_t n = S > 0 ? (size_t)S : 1;
    const std::vector<int32_t> b(n, baud);
    const std::vector<int64_t> t(n, ts_cycles);
    return afsk_tx_streams_create_each(device, S, b.data(), t.data(), h);
}

int afsk_tx_streams_configure(AfskTxStreams *H, int n, const int32_t *h_streams, const int32_t *h_baud, const int64_t *h_ts_cycles)
{
    const char *fn = "afsk_tx_streams_configure";
    if (!H || n < 0 || n > H->S || (n > 0 && (!h_streams || !h_baud || !h_ts_cycles))) { afsk_set_error("%s: bad argument", fn); return AFSK_E_ARG; }
    std::vector<uint8_t> seen((size_t)H->S, 0);
    for (int i = 0; i < n; i++) {
        const int s = h_streams[i];
        if (s < 0 || s >= H->S) { afsk_set_error("%s: stream %d out of range", fn, s); return AFSK_E_ARG; }
        if (seen[s]) { afsk_set_error("%s: stream %d listed twice", fn, s); return AFSK_E_ARG; }
        seen[s] = 1;
    }
    int bf, ml, sl;
    for (int i = 0; i < n; i++)
        if (!afsk_tone_geometry(h_baud[i], &bf, &ml, &sl)) {
            afsk_set_error("Invalid baud rate. (%s: channel %d, baud %d)", fn, h_streams[i], h_baud[i]);
            return AFSK_E_BAUD;
        }
    return tx_streams_call(H, [&] {
        for (int i = 0; i < n; i++) {
            const int s = h_streams[i];
            afsk_tone_geometry(h_baud[i], &bf, &ml, &sl);
            H->baud[s] = h_baud[i]; H->bf[s] = bf; H->ml[s] = ml;
            H->ts_cycles[s] = h_ts_cycles[i] < 0 ? 0 : h_ts_cycles[i];
        }
        return AFSK_OK;
    });
}

int afsk_tx_streams_send(AfskTxStreams *H, int n, const int32_t *h_stream, const int64_t *h_pay_off, const uint8_t *h_payload,
                         int64_t *h_start, int64_t *h_end)
{
    if (!H || n < 0 || (n > 0 && (!h_stream || !h_pay_off || !h_start || !h_end))) {
        afsk_set_error("afsk_tx_streams_send: bad argument");
        return AFSK_E_ARG;
    }
    if (n > 0 && h_pay_off[0] < 0) { afsk_set_error("afsk_tx_streams_send: negative payload offset"); return AFSK_E_ARG; }
    for (int i = 0; i < n; i++) {
        if (h_stream[i] < 0 || h_stream[i] >= H->S) { afsk_set_error("afsk_tx_streams_send: stream %d out of range", h_stream[i]); return AFSK_E_ARG; }
        if (h_pay_off[i + 1] < h_pay_off[i]) { afsk_set_error("afsk_tx_streams_send: payload offsets decrease at message %d", i); return AFSK_E_ARG; }
    }
    if (n > 0 && h_pay_off[n] > h_pay_off[0] && !h_payload) { afsk_set_error("afsk_tx_streams_send: null payload"); return AFSK_E_ARG; }
    return tx_streams_call(H, [&] { return tx_send_run(H, n, h_stream, h_pay_off, h_payload, h_start, h_end); });
}

int afsk_tx_streams_pull(AfskTxStreams *H, int64_t n_frames, int16_t *dst, int on_device, void *stream)
{
    if (!H || n_frames < 0 || (n_frames > 0 && !dst)) { afsk_set_error("afsk_tx_streams_pull: bad argument"); return AFSK_E_ARG; }
    if (n_frames > (INT64_MAX / 16) / H->S) { afsk_set_error("afsk_tx_streams_pull: S * n_frames overflows"); return AFSK_E_ARG; }
    if (on_device && (reinterpret_cast<uintptr_t>(dst) & 15) != 0) {
        afsk_set_error("afsk_tx_streams_pull: device output must be 16-byte aligned");
        return AFSK_E_ARG;
    }
    if ((((int64_t)H->S * n_frames + 7) / 8 + kWinThreads - 1) / kWinThreads > 0x7FFFFFFFLL) {
        afsk_set_error("afsk_tx_streams_pull: window too large");
        return AFSK_E_ARG;
    }
    return tx_streams_call(H, [&] { return tx_pull_run(H, n_frames, dst, on_device, false, AFSK_SAMPLE_S16, 0, (cudaStream_t)stream); });
}

// the argument checks of an interleaved pull (fn names the entry point in the error)
static int pull_frames_check(const char *fn, AfskTxStreams *H, int64_t n_frames, const void *dst, int format, int64_t row_pitch)
{
    if (!H || n_frames < 0 || (n_frames > 0 && !dst)) { afsk_set_error("%s: bad argument", fn); return AFSK_E_ARG; }
    const int size = afsk_sample_size(format);
    if (!size) { afsk_set_error("%s: unknown sample format %d", fn, format); return AFSK_E_ARG; }
    if (row_pitch < H->S) { afsk_set_error("%s: row_pitch %lld < S = %d", fn, (long long)row_pitch, H->S); return AFSK_E_ARG; }
    if ((reinterpret_cast<uintptr_t>(dst) & (uintptr_t)(size - 1)) != 0) {
        afsk_set_error("%s: dst must be aligned to the sample size (%d bytes)", fn, size);
        return AFSK_E_ARG;
    }
    if (n_frames > (INT64_MAX / 16) / row_pitch) { afsk_set_error("%s: row_pitch * n_frames overflows", fn); return AFSK_E_ARG; }
    if ((int64_t)((H->S + kIlC - 1) / kIlC) * ((n_frames + 8 * kIlV - 1) / (8 * kIlV)) > 0x7FFFFFFFLL) {
        afsk_set_error("%s: window too large", fn);
        return AFSK_E_ARG;
    }
    return AFSK_OK;
}

int afsk_tx_streams_pull_interleaved(AfskTxStreams *H, int64_t n_frames, int16_t *dst, int on_device, void *stream)
{
    const char *fn = "afsk_tx_streams_pull_interleaved";
    const int rc = pull_frames_check(fn, H, n_frames, dst, AFSK_SAMPLE_S16, H ? H->S : 0);
    if (rc != AFSK_OK) return rc;
    if (on_device && (reinterpret_cast<uintptr_t>(dst) & 15) != 0) {
        afsk_set_error("%s: device output must be 16-byte aligned", fn);
        return AFSK_E_ARG;
    }
    return tx_streams_call(H, [&] { return tx_pull_run(H, n_frames, dst, on_device, true, AFSK_SAMPLE_S16, H->S, (cudaStream_t)stream); });
}

int afsk_tx_streams_pull_frames(AfskTxStreams *H, int64_t n_frames, void *dst, int format, int on_device, int64_t row_pitch, void *stream)
{
    const int rc = pull_frames_check("afsk_tx_streams_pull_frames", H, n_frames, dst, format, row_pitch);
    if (rc != AFSK_OK) return rc;
    return tx_streams_call(H, [&] { return tx_pull_run(H, n_frames, dst, on_device, true, format, row_pitch, (cudaStream_t)stream); });
}

int afsk_tx_streams_state(const AfskTxStreams *H, int s, int64_t *pulled, int64_t *busy_until, int64_t *pending)
{
    if (!H || s < 0 || s >= H->S) { afsk_set_error("afsk_tx_streams_state: bad argument"); return AFSK_E_ARG; }
    if (pulled) *pulled = H->P;
    if (busy_until) *busy_until = H->last_end[s];
    if (pending) *pending = (int64_t)H->q[s].size();
    return AFSK_OK;
}

int afsk_tx_streams_arena_bytes(const AfskTxStreams *H, int64_t *bytes)
{
    if (!H || !bytes) return AFSK_E_ARG;
    *bytes = (int64_t)(H->arena_alloc[0] + H->arena_alloc[1] + H->d_scratch_cap + H->out_cap);
    return AFSK_OK;
}

int afsk_tx_streams_counters(const AfskTxStreams *H, int64_t *launches, int64_t *moved_bytes, int64_t *compactions)
{
    if (!H) return AFSK_E_ARG;
    if (launches) *launches = H->n_launches;
    if (moved_bytes) *moved_bytes = H->n_moved;
    if (compactions) *compactions = H->n_compactions;
    return AFSK_OK;
}

int afsk_tx_streams_destroy(AfskTxStreams *H)
{
    if (!H) return AFSK_OK;
    AfskDeviceGuard guard(H->device);
    for (void *p : {(void *)H->arena[0], (void *)H->arena[1], (void *)H->d_scratch, (void *)H->d_out}) cudaFree(p);
    if (H->h_stage) cudaFreeHost(H->h_stage);
    delete H;
    return AFSK_OK;
}

}  // extern "C"
