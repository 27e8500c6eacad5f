// upr_maps.cuh -- storage and arithmetic of the CNN's Retinex maps, shared by the recombination kernels (upr_pointwise.cu) and
// the fused Retinex prologue of the CLAHE histogram kernels (upr_clahe.cu).
//
// The illumination map illu (dtype TI) and the enhancement map e (dtype TE) are f32, or fp16 / bf16 when the model runs under
// autocast.  The real network under CUDA autocast emits TI = f32 (ResidualIENet adds the f32 scalar mean(x) to its fp16 head)
// and TE = the autocast dtype, so the two dtypes are independent.  Every map value is widened to f32 on load;
// rnd<T>(v) = f(T(v)) is the rounding torch applies when an op's result has dtype T.  What torch eager evaluates, and so what
// every kernel here evaluates (each step one IEEE f32 operation, no FMA):
//   d = TI(f(illu) + eps);  R = x / f(d);  c = f(e)*f(e), rounded to TE unless under autocast;  enh = R*f(e) + (1-R)*f(c)
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "upr_common.cuh"

namespace upr {

template <typename T> struct MapIO;

template <> struct MapIO<float> {
    using Raw4 = float4;   // 4 pixels as loaded
    static __device__ __forceinline__ float wide(float v) { return v; }
    static __device__ __forceinline__ float narrow(float v) { return v; }
    static __device__ __forceinline__ float ld1(const float* p, uint64_t pol) { return ld_stream_f1(p, pol); }
    static __device__ __forceinline__ float4 ld4raw(const float* p, uint64_t pol) { return ld_stream_f4(p, pol); }
    // no L2 policy operand: the CLAHE histogram kernel keeps its registers for the Lab arithmetic
    static __device__ __forceinline__ float4 ld4nc(const float4* p)
    {
        float4 v;
        asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
        return v;
    }
    static __device__ __forceinline__ float4 wide4(float4 v) { return v; }
    static __device__ __forceinline__ float4 ld4(const float* p, uint64_t pol) { return ld_stream_f4(p, pol); }
    static __device__ __forceinline__ void st4(float* p, float4 v, uint64_t pol) { st_stream_f4(p, v, pol); }
};

__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ __half from_f32(float v, const __half*) { return __float2half_rn(v); }
__device__ __forceinline__ __nv_bfloat16 from_f32(float v, const __nv_bfloat16*) { return __float2bfloat16_rn(v); }
__device__ __forceinline__ __half from_bits(uint32_t b, const __half*) { return __ushort_as_half((unsigned short)b); }
__device__ __forceinline__ __nv_bfloat16 from_bits(uint32_t b, const __nv_bfloat16*) { return __ushort_as_bfloat16((unsigned short)b); }
__device__ __forceinline__ uint32_t to_bits(__half v) { return __half_as_ushort(v); }
__device__ __forceinline__ uint32_t to_bits(__nv_bfloat16 v) { return __bfloat16_as_ushort(v); }

template <typename H> struct MapIO16 {   // H = __half or __nv_bfloat16
    using Raw4 = uint2;    // kept packed until use: fewer registers live across the division slow path
    static __device__ __forceinline__ float wide(H v) { return to_f32(v); }
    static __device__ __forceinline__ H narrow(float v) { return from_f32(v, (const H*)nullptr); }
    static __device__ __forceinline__ float lo(uint32_t u) { return to_f32(from_bits(u & 0xffffu, (const H*)nullptr)); }
    static __device__ __forceinline__ float hi(uint32_t u) { return to_f32(from_bits(u >> 16, (const H*)nullptr)); }
    static __device__ __forceinline__ uint32_t pack(float a, float b) { return to_bits(narrow(a)) | (to_bits(narrow(b)) << 16); }
    static __device__ __forceinline__ float ld1(const H* p, uint64_t pol)
    {
        unsigned short v;
        asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u16 %0, [%1], %2;" : "=h"(v) : "l"(p), "l"(pol));
        return to_f32(from_bits(v, (const H*)nullptr));
    }
    // 4 pixels = 8 bytes: one 64-bit streaming access
    static __device__ __forceinline__ uint2 ld4raw(const H* p, uint64_t pol)
    {
        uint2 v;
        asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.u32 {%0,%1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(p), "l"(pol));
        return v;
    }
    static __device__ __forceinline__ uint2 ld4nc(const uint2* p)
    {
        uint2 v;
        asm("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
        return v;
    }
    static __device__ __forceinline__ float4 wide4(uint2 v) { return make_float4(lo(v.x), hi(v.x), lo(v.y), hi(v.y)); }
    static __device__ __forceinline__ float4 ld4(const H* p, uint64_t pol) { return wide4(ld4raw(p, pol)); }
    static __device__ __forceinline__ void st4(H* p, float4 v, uint64_t pol)
    {
        asm volatile("st.global.L1::no_allocate.L2::cache_hint.v2.u32 [%0], {%1,%2}, %3;" ::"l"(p), "r"(pack(v.x, v.y)),
                     "r"(pack(v.z, v.w)), "l"(pol)
                     : "memory");
    }
};
template <> struct MapIO<__half> : MapIO16<__half> {};
template <> struct MapIO<__nv_bfloat16> : MapIO16<__nv_bfloat16> {};

template <typename T> __device__ __forceinline__ float rnd(float v) { return MapIO<T>::wide(MapIO<T>::narrow(v)); }

// e^2 with the map dtype T: torch rounds pow's result to T, except under CUDA autocast, where pow runs in fp32
template <typename T, bool kAutocast> __device__ __forceinline__ float square(float e)
{
    return kAutocast ? __fmul_rn(e, e) : rnd<T>(__fmul_rn(e, e));
}

// d = TI(f(illu) + eps): torch adds the scalar in fp32 and stores a TI tensor (no rounding for TI = f32)
template <typename TI> __device__ __forceinline__ float illu_eps(float illu, float eps) { return rnd<TI>(__fadd_rn(illu, eps)); }

// R and enhanced of one pixel and channel; TE = e's dtype
template <typename TE, bool kAutocast>
__device__ __forceinline__ void recombine1(float x, float d, float e, float& r, float& o)
{
    r = __fdiv_rn(x, d);
    o = __fadd_rn(__fmul_rn(r, e), __fmul_rn(__fsub_rn(1.0f, r), square<TE, kAutocast>(e)));
}

template <typename T> static inline bool aligned4px(const T* p)
{
    return (reinterpret_cast<uintptr_t>(p) & (4 * sizeof(T) - 1)) == 0;
}

// ---- host: the (illu dtype, e dtype, autocast) triples of the typed entries ----------------------------------------------
// illu_dt in {UPR_DT_F32, e_dt}, e_dt in {F32, F16, BF16}, flags in {0, UPR_RETINEX_AUTOCAST}.  f32 / f32 is one case whatever
// the flag (e*e is f32 either way).
inline bool valid_map_dtypes(int illu_dt, int e_dt, int flags)
{
    return e_dt >= UPR_DT_F32 && e_dt <= UPR_DT_BF16 && (illu_dt == UPR_DT_F32 || illu_dt == e_dt) &&
           (flags & ~UPR_RETINEX_AUTOCAST) == 0;
}

template <typename T> struct MapType { using type = T; };

// Calls f(MapType<TI>, MapType<TE>, std::integral_constant<bool, AC>) for a triple that valid_map_dtypes accepted.
template <typename F> int with_map_types(int illu_dt, int e_dt, int flags, F&& f)
{
    using AcOn = std::integral_constant<bool, true>;
    using AcOff = std::integral_constant<bool, false>;
    const bool ac = flags & UPR_RETINEX_AUTOCAST;
    const bool same = illu_dt == e_dt;
    switch (e_dt) {
    case UPR_DT_F16:
        if (same) return ac ? f(MapType<__half>{}, MapType<__half>{}, AcOn{}) : f(MapType<__half>{}, MapType<__half>{}, AcOff{});
        return ac ? f(MapType<float>{}, MapType<__half>{}, AcOn{}) : f(MapType<float>{}, MapType<__half>{}, AcOff{});
    case UPR_DT_BF16:
        if (same)
            return ac ? f(MapType<__nv_bfloat16>{}, MapType<__nv_bfloat16>{}, AcOn{})
                      : f(MapType<__nv_bfloat16>{}, MapType<__nv_bfloat16>{}, AcOff{});
        return ac ? f(MapType<float>{}, MapType<__nv_bfloat16>{}, AcOn{}) : f(MapType<float>{}, MapType<__nv_bfloat16>{}, AcOff{});
    default: return f(MapType<float>{}, MapType<float>{}, AcOff{});
    }
}

}  // namespace upr
