/*
 * afsk_b200.h — C ABI of libafsk_b200.so, the B200 (sm_100a) batch AFSK modem core.
 *
 * The reference (lavajuno/afskmodem, one pure-Python file) has no FFI/plugin interface; its
 * boundary is the Python class API (afskmodem.py:275-276 Receiver, :420 load, :437 Transmitter,
 * :481 save).  This header is the C surface a binding for that path needs: plain pointers and
 * sizes, no torch types.  Each entry point names the reference function(s) it replaces.
 * INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error (AFSK_E_*); afsk_last_error() gives text
 *     (thread-local).  Nothing throws.  There is NO CPU fallback: without a CUDA device every
 *     compute entry point returns AFSK_E_CUDA.
 *   - device pointers are caller-owned; `stream` is a cudaStream_t passed as void* (NULL =
 *     default stream).  Calls taking a stream are asynchronous on it.
 *   - sample buffers are int16 little-endian, 48 kHz mono, captures concatenated; offsets are in
 *     samples (CSR: capture c = [off[c], off[c+1]) ).  The device sample pointer must be 16-byte
 *     aligned and the allocation must extend to the next 16-byte boundary past off[B].
 *   - one process/thread per GPU; a plan belongs to the device it was created on.
 */
#ifndef AFSK_B200_H
#define AFSK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AFSK_ABI_VERSION 2

/* return codes */
#define AFSK_OK 0
#define AFSK_E_ARG (-1)     /* bad argument (null, misaligned, negative size ...) */
#define AFSK_E_CUDA (-2)    /* CUDA runtime error / no device                      */
#define AFSK_E_BAUD (-3)    /* Exception("Invalid baud rate.")  afskmodem.py:69-70,81-82 */
#define AFSK_E_UNSUPPORTED (-4)

/* per-capture decode status (AfskRxResult.status) */
#define AFSK_ST_OK 0            /* >= 1 coded bit decoded                                      */
#define AFSK_ST_NO_CLOCK 1      /* len(frames) < 4096: "Failed to recover clock" :323-325      */
#define AFSK_ST_NO_DATA 2       /* clock found but 0 bits: "No data." :422-424                 */
#define AFSK_ST_EXC_WAVELEN (-1)/* Exception("Comparing two waveforms of different lengths.")  */
#define AFSK_ST_EXC_INDEX (-2)  /* IndexError at scan_diffs[0] :332 (2*bit_frames >= 4096)      */
#define AFSK_ST_EXC_BAUD (-3)   /* constructor would raise "Invalid baud rate."                */

/* One per capture; the four integers are the reference's debug-log stage values
 * (afskmodem.py:338, :368, :380, :427). */
typedef struct AfskRxResult {
    int32_t status;
    int32_t clock;       /* -1 when no clock */
    int64_t train_end;   /* -1 when no clock */
    int64_t nbits;
    int64_t nbytes;
} AfskRxResult;

typedef struct AfskRxPlan AfskRxPlan;
typedef struct AfskTxPlan AfskTxPlan;

/* ---------------------------------------------------------------- library / device ---- */
int afsk_abi_version(void);
const char *afsk_last_error(void);
int afsk_device_count(int *count);
/* SM count, global memory bytes, compute capability major*10+minor of `device` */
int afsk_device_info(int device, int *sm_count, size_t *mem_bytes, int *cc);

/* minimal memory / stream helpers so a host binding needs no other CUDA wrapper */
int afsk_malloc(int device, size_t bytes, void **dptr);
int afsk_free(int device, void *dptr);
int afsk_host_alloc(size_t bytes, void **hptr);           /* pinned */
int afsk_host_free(void *hptr);
int afsk_memcpy_h2d(int device, void *dst, const void *src, size_t bytes, void *stream);
int afsk_memcpy_d2h(int device, void *dst, const void *src, size_t bytes, void *stream);
int afsk_memset(int device, void *dst, int value, size_t bytes, void *stream);
int afsk_stream_create(int device, void **stream);
int afsk_stream_destroy(int device, void *stream);
int afsk_stream_sync(int device, void *stream);
/* everything enqueued on `waiter` after this call runs after everything enqueued on `signaller`
 * before it (event record + stream wait): lets a copy stream feed a compute stream chunk by chunk */
int afsk_stream_wait_stream(int device, void *waiter, void *signaller);

/* ---------------------------------------------------------------- tone tables ---------- */
/* Waveforms.getSpaceTone / getMarkTone lengths (afskmodem.py:68-85) and Receiver.__bit_frames
 * (:277).  Returns AFSK_E_BAUD where the reference constructor raises. */
int afsk_tone_lengths(int baud, int *bit_frames, int *mark_len, int *space_len);

/* ---------------------------------------------------------------- receiver ------------- */
/*
 * Replaces Receiver.load's compute (afskmodem.py:420-430): __decodeBits :354-381
 * (__recoverClockIndex :322-339, __decodeBit :342-351 with __amplify :287-296 and
 * Waveforms.getDiff/getAmplitude :94-107, __scanTraining :386-390), ECC.decode :154-163 and
 * __bitsToBytes :393-399, for B independent captures.
 *
 * h_offsets[B+1] (samples), h_baud[B], h_amp_end[B] are HOST arrays describing the batch
 * (amp_end = Receiver's amp_end_threshold; amp_start is unused on the file path, :375 vs :306).
 * A plan holds the device-side descriptors and scratch (bit planes, clock indices).
 */
int afsk_rx_plan_create(int device, int B, const int64_t *h_offsets, const int32_t *h_baud,
                        const int32_t *h_amp_end, AfskRxPlan **plan);
/* same, for captures given as arbitrary (possibly non-adjacent) [start, start + len) ranges of one
 * sample buffer — e.g. the recordings afsk_rx_gate_multi cuts out of a long stream */
int afsk_rx_plan_create_ranges(int device, int B, const int64_t *h_start, const int64_t *h_len,
                               const int32_t *h_baud, const int32_t *h_amp_end, AfskRxPlan **plan);
/* Re-targets an existing plan at another batch layout (a drop-in Receiver.load sees a different file
 * length on every call): same arguments as afsk_rx_plan_create_ranges, or h_len == NULL with CSR
 * h_start[B+1].  The plan's device arena is reused when large enough (it only grows), so the call costs
 * one host-to-device copy of the descriptors and no allocation.  Output offsets / launch counts queried
 * earlier are invalidated. */
int afsk_rx_plan_reset(AfskRxPlan *plan, int B, const int64_t *h_start, const int64_t *h_len,
                       const int32_t *h_baud, const int32_t *h_amp_end);
int afsk_rx_plan_destroy(AfskRxPlan *plan);
/* tuning / test switches of a plan; results never depend on them */
#define AFSK_OPT_FRAME_KERNEL 1 /* framing kernel: 0 automatic (by capture length), 1 k_frame_warp (one warp per
                                   capture), 2 k_frame<128,4>, 3 k_frame<512,8>, 4 k_frame<512,8> with 64-bit window
                                   indices (automatic from 2^30 windows per capture).  A variant that cannot
                                   represent the batch is replaced by the automatic choice. */
#define AFSK_OPT_L2_HINT 2      /* L2 evict-first hint on the demodulator's bulk copies: -1 per-kernel default, 0, 1 */
#define AFSK_OPT_FUSED 3        /* schedule of a decode.  0: three kernels (clock, demodulate, frame).  1: auxiliary warps
                                   of the streaming kernel recover the clocks (no k_clock launch).  2: they also frame
                                   every capture as soon as its last tile has retired (one launch per bit length).
                                   -1 automatic = 0 (neither fused level beat the three kernels on a B200, see
                                   profiles/r2_tuning_log.md; both stay available and parity-tested).  Bit lengths over
                                   185 frames (below 260 baud) keep the three kernels; captures of more than 2^18 bit
                                   windows keep the separate framing kernel. */
#define AFSK_OPT_CLOCK_KERNEL 4 /* clock recovery kernel of the three-kernel schedule: 0 (default) automatic = k_clock_q
                                   (32 candidates per thread from registers, no prefix array) for bit lengths of 8..24
                                   frames (6000..2000 baud) and k_clock for the rest; 1 k_clock everywhere (two sweeps
                                   over candidate distances kept in registers); 2 k_clock2 (one sweep with an exact
                                   multiply-shift floor, half the shared memory; bit lengths up to 185 frames, else k_clock) */
#define AFSK_OPT_GROUP_STREAMS 5 /* 1 (default): the demodulator launches of a mixed-baud batch (one per bit length) run on
                                   streams of their own between the clock and framing kernels, so that one group's CTAs
                                   fill the SMs as the previous group's drain; 0: one after the other on the caller's stream */
int afsk_rx_plan_set_option(AfskRxPlan *plan, int option, int value);
/* capacity offsets (bytes, B+1 entries, host memory owned by the plan) of the decoded output */
int afsk_rx_plan_out_offsets(const AfskRxPlan *plan, const int64_t **h_out_off);
/* number of kernel launches one afsk_rx_decode issues for this plan */
int afsk_rx_plan_launches(const AfskRxPlan *plan, int *launches);
/*
 * d_samples: device int16[h_offsets[B]] ; d_out: device bytes[h_out_off[B]] ; d_res: device
 * AfskRxResult[B].  Capture c's payload is d_out[h_out_off[c] .. + d_res[c].nbytes).
 */
int afsk_rx_decode(AfskRxPlan *plan, const int16_t *d_samples, uint8_t *d_out, AfskRxResult *d_res,
                   void *stream);
/*
 * Optional in-line timing of the dominant kernel (k_demod) for roofline reporting: when enabled,
 * every afsk_rx_decode brackets each k_demod launch with CUDA events on the caller's stream.
 * afsk_rx_plan_demod_time synchronizes those events, returns their summed duration and launch
 * count since the last query, and clears them.
 */
int afsk_rx_plan_set_timing(AfskRxPlan *plan, int enable);
int afsk_rx_plan_demod_time(AfskRxPlan *plan, float *ms_total, int *launches);
/* raw decision / quiet flags of capture c after a decode, for diagnostics and stage-level parity
 * tests: d_planes points at interleaved uint32 pairs {bits, quiet}; window k of the capture is
 * bit (k & 31) of pair k >> 5 (LSB first).  *max_windows counts the windows at clock 0; a decode decides
 * the K = #{k >= 0 : clock + k * bit length < n - bit length} windows at the capture's clock, in every
 * schedule and layout, and writes 0 (bit and quiet) for windows K .. of the pair holding window K - 1.  Later
 * pairs are undefined. */
int afsk_rx_plan_planes(const AfskRxPlan *plan, int capture, const uint32_t **d_planes, int64_t *max_windows);
/*
 * Host-buffer convenience (what a drop-in Receiver.load calls): H2D, decode, D2H on `device`.
 * h_out_off[B+1] are capacity offsets into h_out (use afsk_rx_out_capacity per capture).
 * Calls on one device are serialised; the plan and buffers of the previous call are reused.
 */
int afsk_rx_decode_host(int device, const int16_t *h_samples, const int64_t *h_offsets, int B,
                        const int32_t *h_baud, const int32_t *h_amp_end, uint8_t *h_out,
                        const int64_t *h_out_off, AfskRxResult *h_res);
/* afsk_rx_decode_host keeps a plan and grow-only device / pinned buffers per device between calls;
 * this releases them (also done at process exit by the driver) */
int afsk_rx_host_release(int device);
/* upper bound on decoded bytes of a capture of n samples at `baud` */
int64_t afsk_rx_out_capacity(int64_t n_samples, int baud);

/*
 * Receiver.__listen gate arithmetic (afskmodem.py:299-319) over S recorded streams: chunk 0 is
 * discarded, the first 2048-frame chunk with floor(sum|x|/2048) > amp_start opens the recording,
 * it extends through the first chunk with amplitude < amp_end.  h_offsets[S+1] in samples.
 * d_range receives int64 {recorded(0/1), start, end} per stream.  Finite-stream conventions:
 * exhausted before opening → recorded = 0; exhausted before closing → end = last full chunk.
 */
int afsk_rx_gate(int device, const int16_t *d_samples, const int64_t *h_offsets, int S, int amp_start,
                 int amp_end, int64_t timeout_frames, int64_t *d_range, void *stream);

/*
 * Successive Receiver.receive(timeout) calls of ONE receiver over each recorded stream (the
 * reference keeps its input stream open between calls, afskmodem.py:283, so call k+1 starts at the
 * chunk after call k's last read): per call one int64 triple {recorded(0 = "Timed out."), start, end}
 * in d_ranges[s * max_calls * 3 ...], calls made per stream in d_counts[s].  A call that reaches
 * the end of the recording before opening or timing out is not reported.
 */
int afsk_rx_gate_multi(int device, const int16_t *d_samples, const int64_t *h_offsets, int S, int amp_start,
                       int amp_end, int64_t timeout_frames, int max_calls, int64_t *d_ranges,
                       int32_t *d_counts, void *stream);

/*
 * Streaming receiver: S channels, each one Receiver calling receive(timeout) again and again on its own
 * open input stream (afskmodem.py:283, 299-319, 402-417), fed piece by piece as the audio arrives.
 * Chunks lie on the grid of stream frames 2048*k from the first frame pushed to the channel; a partial
 * chunk at the end of a push waits for the next one.  A push returns the receive() calls that became
 * final with it, decoded: calls that timed out (all their ceil(timeout / 2048) chunks present, none
 * loud) and recordings whose closing quiet chunk is present.  A recording without one yet is pending:
 * its samples stay on the device.  For every way of cutting a stream into pushes, the events of all
 * pushes and of afsk_rx_streams_finish are the calls afsk_rx_gate_multi reports over the whole stream.
 * Positions are int64 stream frames.
 */
typedef struct AfskRxStreams AfskRxStreams;
typedef struct AfskRxStreamEvent {      /* 32 bytes, one per final receive() call */
    int32_t stream, recorded;           /* recorded 0 = "Timed out." */
    int64_t call;                       /* index of the call on its channel */
    int64_t start, end;                 /* stream frames of the recording */
} AfskRxStreamEvent;
/* channel s is a Receiver(h_baud[s], h_amp_start[s], h_amp_end[s]) calling receive() with a timeout of
 * h_timeout_frames[s] frames (>= 0): baud / amp_end as for afsk_rx_plan_create, amp_start / timeout_frames as for
 * afsk_rx_gate_multi.  AFSK_E_BAUD where the reference constructor raises (afsk_last_error names the channel). */
int afsk_rx_streams_create_each(int device, int S, const int32_t *h_baud, const int32_t *h_amp_start,
                                const int32_t *h_amp_end, const int64_t *h_timeout_frames, AfskRxStreams **h);
/* the same settings on every channel (a timeout below 0 counts as 0) */
int afsk_rx_streams_create(int device, int S, int baud, int amp_start, int amp_end, int64_t timeout_frames,
                           AfskRxStreams **h);
/* samples: the S pieces concatenated, h_offsets[S+1] (CSR, any length including 0); on_device != 0: a
 * device pointer (16-byte aligned, allocation extending to the next 16-byte boundary past h_offsets[S]),
 * else host memory (pinned recommended).  Synchronizes `stream`.  A bad argument returns AFSK_E_ARG and
 * changes nothing; after any other error the handle refuses every later push / finish (AFSK_E_CUDA) and
 * can only be destroyed. */
int afsk_rx_streams_push(AfskRxStreams *h, const int16_t *samples, int on_device, const int64_t *h_offsets,
                         void *stream, int64_t *n_events);
/* afsk_rx_streams_push of n_frames frames of every channel, given interleaved as a sound card delivers them:
 * frames[f * S + s] = frame f of channel s (n_frames * S samples, frame-major).  Device and host pointers, the
 * host copy and errors as for afsk_rx_streams_push; AFSK_E_ARG also for a negative n_frames, a NULL frames with
 * n_frames > 0 or an n_frames * S that overflows.  Events, state, counters and arena bytes are those of the
 * planar push of the same pieces. */
int afsk_rx_streams_push_interleaved(AfskRxStreams *h, const int16_t *frames, int on_device, int64_t n_frames,
                                     void *stream, int64_t *n_events);
/* sample formats of afsk_rx_streams_push_frames / afsk_tx_streams_pull_frames, each defined by its conversion to
 * and from the int16 samples the modem works on:
 *   S16  int16     receive x                                        transmit s
 *   S32  int32     receive x >> 16 (arithmetic: the top 16 bits)   transmit s << 16
 *   F32  float32   receive clamp(rint(x * 32768), -32768, 32767)    transmit s / 32768 (exact)
 *                  (round half to even, NaN -> 0, +-inf saturate)
 * Transmit then receive is the identity in every format.  Float scales by 32768, not 32767, so that the receive
 * rule is the exact inverse of the transmit rule and -1.0 is -32768. */
#define AFSK_SAMPLE_S16 0
#define AFSK_SAMPLE_S32 1
#define AFSK_SAMPLE_F32 2
/* afsk_rx_streams_push_interleaved of n_frames frames of every channel, read from a window of wider frames:
 * frame f of channel s is element frames[f * row_pitch + s] of the given format (row_pitch >= S, in samples;
 * frames points at row 0's first window sample, aligned to the sample size), converted to int16 by the rule of
 * its format.  Events, state and counters are those of afsk_rx_streams_push_interleaved of the converted,
 * contiguous frames.  Device reads may touch the aligned 16-byte vectors holding window samples, never beyond.
 * A host window is copied packed, in its own format, to the device and converted there.  AFSK_E_ARG (nothing
 * changes) for an unknown format, row_pitch < S, a misaligned pointer, a NULL frames with n_frames > 0, a negative
 * n_frames, an n_frames * row_pitch * size that overflows or a piece too large for one launch. */
int afsk_rx_streams_push_frames(AfskRxStreams *h, const void *frames, int format, int on_device, int64_t n_frames,
                                int64_t row_pitch, void *stream, int64_t *n_events);
/* ends the streams of the n distinct channels h_streams[n] (finite-stream conventions of afsk_rx_gate_multi: a
 * pending recording ends at the last full chunk, a call that has neither opened nor timed out is dropped, a
 * partial chunk is ignored) and returns their final calls.  Each listed channel's next push is frame 0 of a new
 * stream, whose calls count from 0; with the four settings arrays given (one entry per listed channel, as for
 * afsk_rx_streams_create_each) that stream is received with those settings, with all four NULL with the old
 * ones.  Other channels are untouched.  Synchronizes `stream`; errors as for afsk_rx_streams_push. */
int afsk_rx_streams_finish_some(AfskRxStreams *h, int n, const int32_t *h_streams, const int32_t *h_baud,
                                const int32_t *h_amp_start, const int32_t *h_amp_end, const int64_t *h_timeout_frames,
                                void *stream, int64_t *n_events);
/* afsk_rx_streams_finish_some over every channel, settings kept */
int afsk_rx_streams_finish(AfskRxStreams *h, void *stream, int64_t *n_events);
/* host arrays owned by the handle, valid until the next push / finish: n_events events ordered by
 * (stream, call); per event an AfskRxResult (zero with clock = train_end = -1 for a timed-out call) and
 * payload[payload_off[i] .. + res[i].nbytes) (capacity offsets, n_events + 1 entries) */
int afsk_rx_streams_events(const AfskRxStreams *h, const AfskRxStreamEvent **ev, const AfskRxResult **res,
                           const uint8_t **payload, const int64_t **payload_off);
/* channel s: frames pushed, start of the pending recording (-1: none), frames retained on the device */
int afsk_rx_streams_state(const AfskRxStreams *h, int s, int64_t *pushed, int64_t *pending_start, int64_t *retained);
/* device bytes the handle holds (sample arenas, staging and scratch; the decode plan's own arena aside) */
int afsk_rx_streams_arena_bytes(const AfskRxStreams *h, int64_t *bytes);
/* since creation: kernel launches (decodes included), frames moved to keep retained samples (excluding
 * appends), whole-arena compactions */
int afsk_rx_streams_counters(const AfskRxStreams *h, int64_t *launches, int64_t *moved_frames, int64_t *compactions);
int afsk_rx_streams_destroy(AfskRxStreams *h);
/* Retention modes of a receive handle.  AFSK_RETAIN_SAMPLES (the default) keeps every sample of a pending
 * recording on the device until it ends.  AFSK_RETAIN_BITS demodulates a pending recording as it arrives: once
 * 4096 of its frames are in, its clock is recovered and stored, every push decides its complete 32-window plane
 * words (2 bits per window, in a plane arena with the sample arena's policy), and the channel keeps its samples
 * only from its first undecided window (or its partial chunk, if earlier).  Recordings whose status follows from
 * baud and length keep no samples.  AFSK_RETAIN_PAYLOAD does what AFSK_RETAIN_BITS does and also frames each
 * pending recording with a stored clock as its windows are decided: every push searches the windows that fall in
 * chunks the gate has walked for the terminator, then for the first quiet window, and Hamming-decodes whole bytes
 * in between into a payload slot (a third arena with the same policy, two bytes counting as one sample).  The
 * channel keeps plane words only from the one its search or its next incomplete byte needs; once the first quiet
 * window is found the result is fixed, and it keeps no planes, decides no more windows and keeps samples only from
 * its partial chunk.  A recording whose clock is not stored when it ends is decoded as in AFSK_RETAIN_BITS.  In
 * every mode, events, results and payloads are those of AFSK_RETAIN_SAMPLES; only state's retained frames, the
 * counters and arena_bytes differ. */
#define AFSK_RETAIN_SAMPLES 0
#define AFSK_RETAIN_BITS 1
#define AFSK_RETAIN_PAYLOAD 2
/* before the first push or finish only; AFSK_E_ARG (nothing changed) after it or for an unknown mode.  A bits- or
 * payload-mode push of more than 2^32 frames on one channel returns AFSK_E_ARG and changes nothing. */
int afsk_rx_streams_set_retention(AfskRxStreams *h, int mode);
/* channel s's pending recording in bits or payload mode: its stored clock (-1: not yet, or no recording pending)
 * and the windows decided so far (0 in samples mode; in payload mode it stops growing once the recording's first
 * quiet window after the terminator is found) */
int afsk_rx_streams_pending_bits(const AfskRxStreams *h, int s, int32_t *clock, int64_t *windows);
/* channel s's pending recording in bits or payload mode, for diagnostics and stage-level tests: the plane words it
 * keeps on the device, in afsk_rx_plan_planes' {bits, quiet} pair layout.  The first pair holds windows *first_window ..
 * + 31 (a multiple of 32) of the recording, window k starting at frame pending_start + clock + k * bit length; there
 * are *n_windows of them, up to the windows decided.  0 windows (d_planes NULL) in samples mode, with no recording
 * pending, before its clock is stored, or in payload mode once its result is fixed.  The device pointer is valid
 * until the next push or finish. */
int afsk_rx_streams_pending_planes(const AfskRxStreams *h, int s, const uint32_t **d_planes, int64_t *first_window,
                                   int64_t *n_windows);
/* since creation: plane words moved to keep pending recordings' planes, and whole plane-arena compactions (both
 * 0 in samples mode) */
int afsk_rx_streams_plane_counters(const AfskRxStreams *h, int64_t *moved_words, int64_t *compactions);
/* channel s's pending recording in payload mode, as framed so far: *train_end = clock + k0 * bit length once the
 * terminator was seen (-1 before), *nbits the coded bits framed since k0, *ended 1 once the first quiet window at
 * or after k0 was found (the result is then fixed), and its first min(cap, *nbytes) decoded bytes copied to out
 * (out may be NULL when cap is 0).  -1 / 0 / 0 / 0 in other modes, with no recording pending, or before its clock
 * is stored.  Synchronous (one device-to-host copy); AFSK_E_ARG for a NULL handle or pointer, a negative cap or
 * an s out of range. */
int afsk_rx_streams_pending_payload(const AfskRxStreams *h, int s, int64_t *train_end, int64_t *nbits, int32_t *ended,
                                    uint8_t *out, int64_t cap, int64_t *nbytes);
/* since creation: payload bytes moved to keep pending recordings' decoded bytes, and whole payload-arena
 * compactions (both 0 in the other modes) */
int afsk_rx_streams_payload_counters(const AfskRxStreams *h, int64_t *moved_bytes, int64_t *compactions);

/* ---------------------------------------------------------------- transmitter ---------- */
/* frames Transmitter.save writes for a payload of n bytes (afskmodem.py:452-469 then :239-244).
 * Needs the payload only when mark/space tone lengths differ (e.g. 4800 baud); pass NULL else. */
int64_t afsk_tx_num_samples(int baud, int64_t ts_cycles, int64_t payload_bytes, const uint8_t *payload);
/*
 * Replaces Transmitter.__getFrames (:452-469: __bytesToBits :446-450, ECC.encode :166-175,
 * training sequence, terminator, 4800-frame tail) + SoundOutput.__convertFrames (:239-244) for
 * B payloads.  h_pay_off[B+1] bytes; h_baud[B]; h_ts_cycles[B] = int(baud*training_time/2) (:438).
 */
int afsk_tx_plan_create(int device, int B, const int64_t *h_pay_off, const int32_t *h_baud,
                        const int64_t *h_ts_cycles, const uint8_t *h_payload, AfskTxPlan **plan);
int afsk_tx_plan_destroy(AfskTxPlan *plan);
/* sample offsets (B+1, host, owned by the plan; each capture starts on a multiple of 8 samples) */
int afsk_tx_plan_out_offsets(const AfskTxPlan *plan, const int64_t **h_out_off, const int64_t **h_out_len);
int afsk_tx_synth(AfskTxPlan *plan, const uint8_t *d_payload, int16_t *d_out, void *stream);
int afsk_tx_synth_host(int device, const uint8_t *h_payload, const int64_t *h_pay_off, int B,
                       const int32_t *h_baud, const int64_t *h_ts_cycles, int16_t *h_out,
                       const int64_t *h_out_off);

/*
 * Streaming transmitter: S channels, each one Transmitter whose output stream stays open, calling
 * transmit(data) again and again (afskmodem.py:472-478 hands __getFrames to SoundOutput.play, :247-252,
 * which writes what save() writes).  The channels share one timeline of frames, pulled in windows like
 * the periods of a multi-channel sound card; P = frames pulled so far.  A message sent to channel s starts
 * at max(P, end of s's last message) and lasts afsk_tx_num_samples frames (always even); its frames are
 * exactly save()'s, every frame outside a message is 0.  The device keeps payload bytes only (plus, for
 * unequal tone lengths, each message's codeword start table); every pull synthesizes its window from them.
 */
typedef struct AfskTxStreams AfskTxStreams;
/* channel s is a Transmitter with h_baud[s] / h_ts_cycles[s] (as for afsk_tx_plan_create); AFSK_E_BAUD where the
 * reference constructor raises (afsk_last_error names the channel) */
int afsk_tx_streams_create_each(int device, int S, const int32_t *h_baud, const int64_t *h_ts_cycles, AfskTxStreams **h);
/* the same settings on every channel */
int afsk_tx_streams_create(int device, int S, int baud, int64_t ts_cycles, AfskTxStreams **h);
/* messages sent from now on to the n distinct channels h_streams[n] use h_baud[i] / h_ts_cycles[i]; messages
 * already queued keep theirs.  A bad argument returns AFSK_E_ARG (AFSK_E_BAUD for a baud the reference
 * constructor rejects) and changes nothing. */
int afsk_tx_streams_configure(AfskTxStreams *h, int n, const int32_t *h_streams, const int32_t *h_baud,
                              const int64_t *h_ts_cycles);
/* queues n messages (message i = h_payload[h_pay_off[i] .. h_pay_off[i+1]) on channel h_stream[i], in order)
 * and returns their timeline frames [h_start[i], h_end[i]).  Synchronous. */
int afsk_tx_streams_send(AfskTxStreams *h, int n, const int32_t *h_stream, const int64_t *h_pay_off,
                         const uint8_t *h_payload, int64_t *h_start, int64_t *h_end);
/* the next n_frames frames of every channel as an S x n_frames row-major int16 array: on_device != 0, a
 * 16-byte aligned device pointer, else host memory (pinned recommended); nothing past S * n_frames is
 * written.  Synchronizes `stream`.  A bad argument returns AFSK_E_ARG and changes nothing; after any other
 * error the handle refuses every later send / pull (AFSK_E_CUDA) and can only be destroyed. */
int afsk_tx_streams_pull(AfskTxStreams *h, int64_t n_frames, int16_t *dst, int on_device, void *stream);
/* afsk_tx_streams_pull with the window written interleaved, as a sound card takes it: dst[f * S + s] = frame f
 * of channel s (n_frames x S, frame-major), the transpose of afsk_tx_streams_pull's array; nothing past
 * S * n_frames is written.  Arguments and errors as for afsk_tx_streams_pull. */
int afsk_tx_streams_pull_interleaved(AfskTxStreams *h, int64_t n_frames, int16_t *dst, int on_device, void *stream);
/* afsk_tx_streams_pull_interleaved into a window: dst[f * row_pitch + s] = frame f of channel s, converted by the
 * rule of format (AFSK_SAMPLE_*; dst aligned to the sample size, row_pitch >= S).  Nothing outside the window's
 * n_frames x S elements is written, so handles may write disjoint windows of one buffer.  Host output is
 * synthesized packed on the device and copied out row by row.  Errors as for afsk_rx_streams_push_frames. */
int afsk_tx_streams_pull_frames(AfskTxStreams *h, int64_t n_frames, void *dst, int format, int on_device,
                                int64_t row_pitch, void *stream);
/* channel s: frames pulled (P), end of its last message sent (<= P: idle), messages not yet fully pulled */
int afsk_tx_streams_state(const AfskTxStreams *h, int s, int64_t *pulled, int64_t *busy_until, int64_t *pending);
/* device bytes the handle holds (payload arenas, descriptors, host-output staging) */
int afsk_tx_streams_arena_bytes(const AfskTxStreams *h, int64_t *bytes);
/* since creation: kernel launches, arena bytes moved by compactions, compactions */
int afsk_tx_streams_counters(const AfskTxStreams *h, int64_t *launches, int64_t *moved_bytes, int64_t *compactions);
int afsk_tx_streams_destroy(AfskTxStreams *h);

/* ---------------------------------------------------------------- wav files ------------ */
/*
 * Host ingest / egress for batches of files (one pool of host threads; threads <= 0: all cores).
 * Replaces SoundInput.loadFromFile + __convertFrames (afskmodem.py:201-205, 213-217: every frame byte
 * of the data chunk, paired little-endian signed whatever the header says about channels or sample
 * width) and SoundOutput.writeToFile (afskmodem.py:256-263: 1 channel / 2 bytes / 48000 Hz).
 * Per-file status: AFSK_WAV_OK, or a reason to hand the file to CPython's wave module instead
 * (which then raises exactly what the reference raises).
 */
#define AFSK_WAV_OK 0
#define AFSK_WAV_E_OPEN 1      /* cannot open / read / write the file                     */
#define AFSK_WAV_E_FORMAT 2    /* not plain RIFF/WAVE PCM with fmt before data            */
/* samples (= data bytes / 2) and file position of the first frame byte of each file */
int afsk_wav_probe(const char *const *paths, int n, int threads, int64_t *h_nsamples, int64_t *h_data_pos,
                   int32_t *h_status);
/* reads file i's samples into h_dst[h_offsets[i] ...] (pinned memory recommended).  With d_dst != NULL,
 * spans of about span_samples consecutive samples are copied to d_dst (same offsets) on `stream` as
 * soon as their files are in memory, so that reading overlaps the PCIe transfer.
 * h_dst == NULL (d_dst required): the files stream through a process-wide ring of pinned staging slots
 * (span_samples each, 8 MB by default, four slots) straight to the device; no host copy of the corpus is kept, the
 * first call of a process costs what later calls cost, and the call returns once every copy has landed. */
int afsk_wav_load(const char *const *paths, int n, int threads, const int64_t *h_data_pos, const int64_t *h_nsamples,
                  const int64_t *h_offsets, int16_t *h_dst, int device, int16_t *d_dst, int64_t span_samples,
                  void *stream, int32_t *h_status);
/* writes h_src[h_start[i] .. + h_len[i]) as file i, byte-identical to the reference's writeToFile */
int afsk_wav_save(const char *const *paths, int n, int threads, const int16_t *h_src, const int64_t *h_start,
                  const int64_t *h_len, int32_t *h_status);

#ifdef __cplusplus
}
#endif
#endif /* AFSK_B200_H */
