// afsk_common.cuh — shared helpers for libafsk_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/afsk_b200.h"

#define AFSK_RATE 48000
#define AFSK_SYNC_FRAMES 4096     // afskmodem.py:323,327
#define AFSK_GATE_CHUNK 2048      // afskmodem.py:189,209,310
#define AFSK_TAIL_FRAMES 4800     // afskmodem.py:468

void afsk_set_error(const char *fmt, ...);

#define AFSK_CUDA(call)                                                                    \
    do {                                                                                   \
        cudaError_t e__ = (call);                                                          \
        if (e__ != cudaSuccess) {                                                          \
            afsk_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return AFSK_E_CUDA;                                                            \
        }                                                                                  \
    } while (0)

// RAII device switch for the calling host thread
struct AfskDeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit AfskDeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~AfskDeviceGuard() {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
};

// grow-only buffers: reallocated (contents dropped) with a quarter more than asked when `need` exceeds `*cap`
static inline cudaError_t grow_device(void **p, size_t *cap, size_t need)
{
    if (need <= *cap) return cudaSuccess;
    if (*p) cudaFree(*p);
    *p = nullptr; *cap = 0;
    const size_t want = need + need / 4 + 4096;
    const cudaError_t e = cudaMalloc(p, want);
    if (e == cudaSuccess) *cap = want;
    return e;
}
static inline cudaError_t grow_pinned(void **p, size_t *cap, size_t need)
{
    if (need <= *cap) return cudaSuccess;
    if (*p) cudaFreeHost(*p);
    *p = nullptr; *cap = 0;
    const size_t want = need + need / 4 + 4096;
    const cudaError_t e = cudaMallocHost(p, want);
    if (e == cudaSuccess) *cap = want;
    return e;
}

// Tone geometry of a baud rate (Waveforms.getSpaceTone/getMarkTone, afskmodem.py:68-85;
// Receiver.__bit_frames :277).  Returns false where the constructor raises "Invalid baud rate.".
static inline bool afsk_tone_geometry(int baud, int *bf, int *mark_len, int *space_len)
{
    if (baud <= 0 || AFSK_RATE % baud != 0) return false;          // :69-70
    if (AFSK_RATE % (2 * (long long)baud) != 0) return false;      // :83 -> :69-70 at 2*baud
    int bit_frames = AFSK_RATE / baud;
    *bf = bit_frames;
    *space_len = 2 * (bit_frames / 2);                             // int(bf/2) twice
    *mark_len = 4 * ((bit_frames / 2) / 2);                        // two space tones at 2*baud
    return true;
}

// ---- device PTX helpers -------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t afsk_smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));   // volatile: stays behind the barrier
    return v;
}
// predicated shared-memory load: the result is undefined (and the address not touched) when !pred
__device__ __forceinline__ uint32_t lds_u32_if(uint32_t addr, bool pred)
{
    uint32_t v;
    asm volatile("{\n\t.reg .pred p;\n\t"
        "setp.ne.u32 p, %2, 0;\n\t"
        "@p ld.shared.u32 %0, [%1];\n\t}"
        : "=r"(v)
        : "r"(addr), "r"((uint32_t)pred));
    return v;
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(afsk_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(afsk_smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(afsk_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(afsk_smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    while (!mbar_try_wait(bar, parity)) {
    }
}
// 1-D TMA bulk copy global -> shared (UBLKCP in SASS); src/dst 16-byte aligned, bytes % 16 == 0
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     afsk_smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(afsk_smem_u32(bar))
                 : "memory");
}
// byte permute with the sign-replicate selector bit (the __byte_perm intrinsic masks it off)
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
// same with an L2 evict-first hint: the samples are read exactly once
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_g2s_hint(void *dst, const void *src, uint32_t bytes, uint64_t *bar, uint64_t pol)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     afsk_smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(afsk_smem_u32(bar)), "l"(pol)
                 : "memory");
}
// 16-byte asynchronous copy global -> shared (LDGSTS.BYPASS): the destination is the thread's choice, which is what a
// padded (bank-conflict-free) layout needs and a bulk copy cannot give
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16_hint(uint32_t dst, const void *src, uint64_t pol)
{
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "l"(pol) : "memory");
}
// one arrival on the mbarrier once every cp.async this thread has issued so far has landed (the count is not raised:
// the barrier's expected arrivals include it)
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t *bar)
{
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(afsk_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ uint4 ld_nc_v4(const void *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// the sample-format rules of include/afsk_b200.h (AFSK_SAMPLE_*), element by element.  x * 32768 is exact in float,
// and cvt.rni.s32.f32 rounds half to even, saturates and maps NaN to 0, so the clamp finishes the receive rule.
__device__ __forceinline__ int16_t sample_to_s16(int16_t x) { return x; }
__device__ __forceinline__ int16_t sample_to_s16(int32_t x) { return (int16_t)(x >> 16); }
__device__ __forceinline__ int16_t sample_to_s16(float x) { return (int16_t)min(max(__float2int_rn(x * 32768.f), -32768), 32767); }
template <typename T> __device__ __forceinline__ T sample_from_s16(int16_t s);
template <> __device__ __forceinline__ int16_t sample_from_s16<int16_t>(int16_t s) { return s; }
template <> __device__ __forceinline__ int32_t sample_from_s16<int32_t>(int16_t s) { return (int32_t)((uint32_t)(int32_t)s << 16); }
template <> __device__ __forceinline__ float sample_from_s16<float>(int16_t s) { return (float)s * (1.f / 32768.f); }
#endif

// bytes per sample of an AFSK_SAMPLE_* format, 0 for an unknown one
static inline int afsk_sample_size(int format)
{
    return format == AFSK_SAMPLE_S16 ? 2 : format == AFSK_SAMPLE_S32 || format == AFSK_SAMPLE_F32 ? 4 : 0;
}
