// upr_common.cuh -- shared device/host helpers for the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
#include <mutex>
#include <atomic>
#include <cstdint>

#include "../../include/upretinex_b200.h"

#if defined(__CUDA_ARCH__) && __CUDA_ARCH__ < 1000
#error "upretinex_b200 kernels are written for sm_100a (B200) only"
#endif

#define UPR_CUDA_TRY(expr)                          \
    do {                                            \
        cudaError_t _e = (expr);                    \
        if (_e != cudaSuccess) return int(_e);      \
    } while (0)

#define UPR_LAUNCH_CHECK()                          \
    do {                                            \
        cudaError_t _e = cudaPeekAtLastError();     \
        if (_e != cudaSuccess) return int(_e);      \
    } while (0)

namespace upr {

constexpr int kNumSMsB200 = 148;

// upr_api.cu: two library-owned side streams per device for the chunked two-stream schedules (created on first use, never
// destroyed).  Hold side_pool_mutex() from side_pool() until the join events are recorded.
struct SidePool {
    cudaStream_t s[2] = {nullptr, nullptr};
    cudaEvent_t fork = nullptr, join[2] = {nullptr, nullptr};
    bool ready = false;
};
std::mutex& side_pool_mutex();
SidePool* side_pool();          // nullptr when the streams cannot be created (the caller then runs on its own stream)
// frames per chunk of the chunked schedules (~25 Mpx: 3 x 4K, 12 x 1080p)
inline int chunk_frames(long long plane) { return int(plane >= 25000000LL ? 1 : 25000000LL / plane); }

// The chunked two-stream schedule: launch(f0, nf, stream) enqueues the work of frames [f0, f0 + nf).  With at least two chunks
// of `chunk` frames and a side pool, consecutive chunks go to the two side streams, which fork from s and join back into it
// (graph-capturable); otherwise one launch(0, n, s).  Stops at the first failed launch and returns its status.
template <typename Launch>
int run_chunked(cudaStream_t s, int n, int chunk, Launch&& launch)
{
    if (n >= 2 * chunk) {
        std::lock_guard<std::mutex> guard(side_pool_mutex());
        if (SidePool* pool = side_pool()) {
            UPR_CUDA_TRY(cudaEventRecord(pool->fork, s));
            for (int i = 0; i < 2; ++i) UPR_CUDA_TRY(cudaStreamWaitEvent(pool->s[i], pool->fork, 0));
            int rc = UPR_OK;
            for (int f0 = 0, k = 0; f0 < n && rc == UPR_OK; f0 += chunk, ++k)
                rc = launch(f0, std::min(chunk, n - f0), pool->s[k & 1]);
            for (int i = 0; i < 2; ++i) {      // always join, also after a failed launch: the caller's stream must not run ahead
                UPR_CUDA_TRY(cudaEventRecord(pool->join[i], pool->s[i]));
                UPR_CUDA_TRY(cudaStreamWaitEvent(s, pool->join[i], 0));
            }
            return rc;
        }
    }
    return launch(0, n, s);
}

// upr_pointwise.cu: out = clamp(enh * gain[frame], 0, 1) on stream s (the kernel behind upr_scale_clamp_f32)
int scale_clamp_launch(const float* enh, const float* gain, float* out, int n, int c, int h, int w, cudaStream_t s);

// upr_multiscale.cu: the streaming statistics kernel.  ms_stream_geometry decides once per call whether it serves h x w frames
// at x (h, w multiples of 4 and at least 8, x 16-byte aligned, at most kMsMaxParts row segments x column bands per frame) and
// fills in its band count and segment height; false means the generic multi-kernel path (upr_multiscale_stats_f32).
// ms_stream_launch_range launches it with that geometry for frames [f0, f0 + nf) of a batch of n_total frames on stream s
// (x, means3, gain already point at frame f0; the workspace is the whole batch's).
struct MsStreamGeom {
    int bands, seg_rows;
};
bool ms_stream_geometry(int h, int w, const float* x, MsStreamGeom* geo);
int ms_stream_launch_range(const float* x, int nf, int h, int w, const MsStreamGeom& geo, void* ms_ws, size_t ms_ws_bytes,
                           int n_total, int f0, float* means3, float* gain, cudaStream_t s);

__host__ __device__ inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: a process that drives several GPUs must set it
// on each of them.  `mask` is one bit per device ordinal (benign race: the call is idempotent).
template <typename Kernel>
inline cudaError_t ensure_dynamic_smem(Kernel kernel, size_t bytes, std::atomic<unsigned long long>& mask)
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const unsigned long long bit = 1ull << (dev & 63);
    if (mask.load(std::memory_order_acquire) & bit) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes));
    if (e == cudaSuccess) mask.fetch_or(bit, std::memory_order_release);
    return e;
}
// (plain-word overload for call sites that keep their own function-local static; same benign, idempotent race)
template <typename Kernel>
inline cudaError_t ensure_dynamic_smem(Kernel kernel, size_t bytes, unsigned long long& mask)
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const unsigned long long bit = 1ull << (dev & 63);
    if (mask & bit) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes));
    if (e == cudaSuccess) mask |= bit;
    return e;
}

// ---------------------------------------------------------------------------------------
// streaming global accesses: every f32 pixel is touched exactly once, so keep it out of L1
// and mark it evict-first in L2; the u8 Lab intermediate is what should stay L2-resident.
// ---------------------------------------------------------------------------------------
// (sm_100a accepts the bare .L2::evict_* qualifiers only on 256-bit accesses, so narrower ones
//  carry a createpolicy descriptor through .L2::cache_hint.)
__device__ __forceinline__ uint64_t policy_evict_first()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_last()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ float4 ld_stream_f4(const float* p, uint64_t pol)
{
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ float ld_stream_f1(const float* p, uint64_t pol)
{
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void st_stream_f4(float* p, float4 v, uint64_t pol)
{
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y),
                 "f"(v.z), "f"(v.w), "l"(pol)
                 : "memory");
}
__device__ __forceinline__ void st_stream_f1(float* p, float v, uint64_t pol)
{
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(p), "f"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_hint_u32(void* p, uint32_t v, uint64_t pol)
{
    asm volatile("st.global.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ uint32_t ld_hint_u32(const void* p, uint64_t pol)
{
    uint32_t v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}

// ---------------------------------------------------------------------------------------
// numpy `(x*255).astype(uint8)` (reference adaptive_params.py:142): fp32 multiply, truncate
// toward zero, wrap mod 256; NaN, +-inf and |v| >= 2^31 give 0 (x86 cvttss2si "indefinite").
// cvt.rzi.s32.f32 saturates instead, so only the positive overflow needs a fix-up
// (INT_MIN already has a zero low byte, NaN converts to 0).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ int quantize_u8(float x)
{
    int i = __float2int_rz(__fmul_rn(x, 255.0f));
    i = (i == 0x7fffffff) ? 0 : i;
    return i & 0xff;
}

// ---------------------------------------------------------------------------------------
// save_image's quantiser (enhancers/simple_enhance.py:65-100): (clip(v, 0, 1) * 255).astype(uint8) -- fp32 product,
// truncation.  NaN clips to NaN and casts to 0 on the host; fmaxf(NaN, 0) = 0 gives the same byte here.  One definition for
// upr_quantize_u8_f32 and every epilogue that emits the stored frame itself.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned save_u8(float v)
{
    return unsigned(__float2int_rz(__fmul_rn(fminf(fmaxf(v, 0.0f), 1.0f), 255.0f)));
}
// four bytes of four consecutive pixels of one plane, little-endian
__device__ __forceinline__ unsigned pack4_u8(const unsigned (&q)[4]) { return q[0] | (q[1] << 8) | (q[2] << 16) | (q[3] << 24); }
// four RGB pixels, q[channel][pixel], as the 12 interleaved bytes R0 G0 B0 R1 | G1 B1 R2 G2 | B2 R3 G3 B3 at a 4-byte aligned o
__device__ __forceinline__ void st_rgb4_u8(unsigned char* o, const unsigned (&q)[3][4])
{
    unsigned* o32 = reinterpret_cast<unsigned*>(o);
    o32[0] = q[0][0] | (q[1][0] << 8) | (q[2][0] << 16) | (q[0][1] << 24);
    o32[1] = q[1][1] | (q[2][1] << 8) | (q[0][2] << 16) | (q[1][2] << 24);
    o32[2] = q[2][2] | (q[0][3] << 8) | (q[1][3] << 16) | (q[2][3] << 24);
}

// u8 -> f32 without the (slower) conversion pipe: 0x4B000000 | b is 2^23 + b.
__device__ __forceinline__ float byte_to_float(uint32_t word, int k)
{
    return __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7540 | k)) - 8388608.0f;
}

// ---------------------------------------------------------------------------------------
// Blackwell packed fp32: FFMA2 / FADD2 / FMUL2 process two fp32 lanes per issue slot on an aligned register pair.
// CAUTION: ptxas contracts mul.rn.f32x2 + add/sub.rn.f32x2 into one FFMA2 -- with .rn on both, inside asm volatile and under
// -fmad=false -- so these are only for arithmetic that is exact in fp32 or tolerant of contraction; a mixed-rounding pair
// (mul.rn then add.rz) is left alone.  (profiles/r4_saliency.md)
// ---------------------------------------------------------------------------------------
typedef unsigned long long f32x2;   // (lo, hi) = two fp32 values in an aligned register pair

__device__ __forceinline__ f32x2 pk2(float lo, float hi)
{
    f32x2 r;
    asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(f32x2 v, float& lo, float& hi)
{
    asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c)
{
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ f32x2 fma2_rz(f32x2 a, f32x2 b, f32x2 c)
{
    f32x2 r;
    asm("fma.rz.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b)
{
    f32x2 r;
    // volatile: ptxas contracts mul.rn.f32x2 + add/sub.f32x2 into FFMA2 (observed), which would skip the rounding of x * 255
    asm volatile("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 add2_rz(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm volatile("add.rz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

__device__ __forceinline__ int warp_sum(int v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace upr
