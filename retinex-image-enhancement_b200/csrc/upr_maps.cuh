// upr_maps.cuh -- storage and arithmetic of the CNN's Retinex maps, shared by the recombination kernels (upr_pointwise.cu),
// the fused Retinex prologue of the CLAHE histogram kernels (upr_clahe.cu) and the map epilogues of the content-aware,
// multi-scale and predict inference modes (k_maps_epilogue_*, below).
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

__device__ __forceinline__ float clamp01_keep_nan(float v)
{
    // torch.clamp propagates NaN; fminf/fmaxf would not
    return v < 0.0f ? 0.0f : (v > 1.0f ? 1.0f : v);
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

inline size_t map_dtype_bytes(int dt) { return dt == UPR_DT_F32 ? 4 : 2; }

// ---- map epilogues: the recombination formed in registers inside the last pass of an inference mode ------------------------
// The checked operands of a maps entry: x f32 [n][3][h][w], illu [n][1][h][w] in illu_dt, e [n][3][h][w] in e_dt.  The result
// is either out (f32 [n][3][h][w]) or out8 (u8 [n][h][w][3], the frame save_image stores) with, optionally, illu8
// (u8 [n][h][w][1]) = save_u8(f(illu)), the stored illumination frame.
struct MapsArgs {
    const float* x;
    const void* illu;
    int illu_dt;
    const void* e;
    int e_dt;
    int flags;
    float eps;
    float* out;
    unsigned char* out8;
    unsigned char* illu8;

    // the operands of frames [f0, n) (frames of `plane` pixels)
    MapsArgs at(int f0, long long plane) const
    {
        const long long p1 = f0 * plane, p3 = 3 * p1;
        MapsArgs m = *this;
        m.x = x + p3;
        m.illu = static_cast<const char*>(illu) + p1 * map_dtype_bytes(illu_dt);
        m.e = static_cast<const char*>(e) + p3 * map_dtype_bytes(e_dt);
        m.out = out ? out + p3 : nullptr;
        m.out8 = out8 ? out8 + p3 : nullptr;
        m.illu8 = illu8 ? illu8 + p1 : nullptr;
        return m;
    }
};

// Gain policies of the epilogue: frame(f) gives the per-frame state, whose g4(q) / g1(p) are the gains of pixels 4q .. 4q+3 / p.
// kApply: out = clamp(enh * gain, 0, 1); otherwise out = enh.
struct NoGain {   // predict: the recombined frame itself
    static constexpr bool kApply = false;
    struct Frame {
        __device__ float4 g4(long long) const { return make_float4(1.0f, 1.0f, 1.0f, 1.0f); }
        __device__ float g1(long long) const { return 1.0f; }
    };
    __device__ Frame frame(int) const { return {}; }
};

struct FrameGain {   // multi-scale (multi_scale.py:97-98): one gain per frame
    const float* gain;
    static constexpr bool kApply = true;
    struct Frame {
        float s;
        __device__ float4 g4(long long) const { return make_float4(s, s, s, s); }
        __device__ float g1(long long) const { return s; }
    };
    __device__ Frame frame(int f) const { return {__ldg(gain + f)}; }
};

constexpr int kMapThreads = 256;

// One item = 4 pixels of a frame, all three channels: 128-bit x, 4-pixel map groups (MapIO), f32 out as 128-bit stores or u8 out
// as 12 + 4 bytes (st_rgb4_u8, 4-byte aligned).  Grid (parts, frames): blockIdx.y walks the frames, blockIdx.x the pixels.
template <typename TI, typename TE, bool kAutocast, bool kU8, class Gain>
__global__ void __launch_bounds__(kMapThreads, 1)
k_maps_epilogue_vec(const float* __restrict__ x, const TI* __restrict__ illu, const TE* __restrict__ e, float* __restrict__ out,
                    unsigned char* __restrict__ out8, unsigned char* __restrict__ illu8, int n, long long plane4, float eps,
                    const Gain gain)
{
    const uint64_t pol = policy_evict_first();
    const long long stride = (long long)gridDim.x * kMapThreads;
    for (int f = blockIdx.y; f < n; f += gridDim.y) {
        const typename Gain::Frame gf = gain.frame(f);
        for (long long p = (long long)blockIdx.x * kMapThreads + threadIdx.x; p < plane4; p += stride) {
            const long long o1 = ((long long)f * plane4 + p) * 4, o3 = ((long long)f * 3 * plane4 + p) * 4;
            const float4 il = MapIO<TI>::ld4(illu + o1, pol);
            const float d[4] = {illu_eps<TI>(il.x, eps), illu_eps<TI>(il.y, eps), illu_eps<TI>(il.z, eps), illu_eps<TI>(il.w, eps)};
            float4 xv[3];
            typename MapIO<TE>::Raw4 ev[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                xv[c] = ld_stream_f4(x + o3 + c * plane4 * 4, pol);
                ev[c] = MapIO<TE>::ld4raw(e + o3 + c * plane4 * 4, pol);
            }
            const float4 g = gf.g4(p);
            unsigned q[3][4];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float4 ef = MapIO<TE>::wide4(ev[c]);
                float4 r, o;
                recombine1<TE, kAutocast>(xv[c].x, d[0], ef.x, r.x, o.x);
                recombine1<TE, kAutocast>(xv[c].y, d[1], ef.y, r.y, o.y);
                recombine1<TE, kAutocast>(xv[c].z, d[2], ef.z, r.z, o.z);
                recombine1<TE, kAutocast>(xv[c].w, d[3], ef.w, r.w, o.w);
                if (Gain::kApply) {
                    o.x = clamp01_keep_nan(__fmul_rn(o.x, g.x));
                    o.y = clamp01_keep_nan(__fmul_rn(o.y, g.y));
                    o.z = clamp01_keep_nan(__fmul_rn(o.z, g.z));
                    o.w = clamp01_keep_nan(__fmul_rn(o.w, g.w));
                }
                if (kU8) {
                    q[c][0] = save_u8(o.x);
                    q[c][1] = save_u8(o.y);
                    q[c][2] = save_u8(o.z);
                    q[c][3] = save_u8(o.w);
                } else {
                    st_stream_f4(out + o3 + c * plane4 * 4, o, pol);
                }
            }
            if (kU8) {
                st_rgb4_u8(out8 + o1 * 3, q);
                if (illu8) {
                    const unsigned qi[4] = {save_u8(il.x), save_u8(il.y), save_u8(il.z), save_u8(il.w)};
                    *reinterpret_cast<unsigned*>(illu8 + o1) = pack4_u8(qi);
                }
            }
        }
    }
}

// Any shape and alignment: one item = one pixel of a frame, all three channels.
template <typename TI, typename TE, bool kAutocast, bool kU8, class Gain>
__global__ void __launch_bounds__(kMapThreads)
k_maps_epilogue_scalar(const float* __restrict__ x, const TI* __restrict__ illu, const TE* __restrict__ e, float* __restrict__ out,
                       unsigned char* __restrict__ out8, unsigned char* __restrict__ illu8, int n, long long plane, float eps,
                       const Gain gain)
{
    const long long stride = (long long)gridDim.x * kMapThreads;
    for (int f = blockIdx.y; f < n; f += gridDim.y) {
        const typename Gain::Frame gf = gain.frame(f);
        for (long long p = (long long)blockIdx.x * kMapThreads + threadIdx.x; p < plane; p += stride) {
            const long long o1 = (long long)f * plane + p;
            const float il = MapIO<TI>::wide(illu[o1]);
            const float d = illu_eps<TI>(il, eps);
            const float g = gf.g1(p);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const long long o = ((long long)f * 3 + c) * plane + p;
                float r, v;
                recombine1<TE, kAutocast>(x[o], d, MapIO<TE>::wide(e[o]), r, v);
                if (Gain::kApply) v = clamp01_keep_nan(__fmul_rn(v, g));
                if (kU8) out8[o1 * 3 + c] = (unsigned char)save_u8(v);
                else out[o] = v;
            }
            if (kU8 && illu8) illu8[o1] = (unsigned char)save_u8(il);
        }
    }
}

// The epilogue over n frames of h x w on stream s: the vector kernel when the frame is a whole number of 4-pixel groups and every
// operand is aligned to one, the scalar kernel otherwise.  out8 selects the u8 result.
template <class Gain>
int maps_epilogue(const MapsArgs& m, int n, int h, int w, const Gain& gain, cudaStream_t s)
{
    return with_map_types(m.illu_dt, m.e_dt, m.flags, [&](auto ti, auto te, auto ac) -> int {
        using TI = typename decltype(ti)::type;
        using TE = typename decltype(te)::type;
        constexpr bool AC = decltype(ac)::value;
        const TI* illu = static_cast<const TI*>(m.illu);
        const TE* e = static_cast<const TE*>(m.e);
        const long long plane = (long long)h * w;
        const bool u8 = m.out8 != nullptr;
        const bool vec = plane % 4 == 0 && aligned16(m.x) && aligned4px(illu) && aligned4px(e) &&
                         (u8 ? (reinterpret_cast<uintptr_t>(m.out8) & 3u) == 0 && (reinterpret_cast<uintptr_t>(m.illu8) & 3u) == 0
                             : aligned16(m.out));
        const long long work = vec ? plane / 4 : plane;
        // ~16 CTAs per SM over the whole batch, at least 2 items per thread
        const int parts = int(std::max<long long>(1, std::min<long long>((work + kMapThreads * 2 - 1) / (kMapThreads * 2),
                                                                         (16LL * kNumSMsB200 + n - 1) / n)));
        const dim3 grid(parts, std::min(n, 65535));
        if (vec && u8)
            k_maps_epilogue_vec<TI, TE, AC, true, Gain><<<grid, kMapThreads, 0, s>>>(m.x, illu, e, nullptr, m.out8, m.illu8, n, work, m.eps, gain);
        else if (vec)
            k_maps_epilogue_vec<TI, TE, AC, false, Gain><<<grid, kMapThreads, 0, s>>>(m.x, illu, e, m.out, nullptr, nullptr, n, work, m.eps, gain);
        else if (u8)
            k_maps_epilogue_scalar<TI, TE, AC, true, Gain><<<grid, kMapThreads, 0, s>>>(m.x, illu, e, nullptr, m.out8, m.illu8, n, work, m.eps, gain);
        else
            k_maps_epilogue_scalar<TI, TE, AC, false, Gain><<<grid, kMapThreads, 0, s>>>(m.x, illu, e, m.out, nullptr, nullptr, n, work, m.eps, gain);
        UPR_LAUNCH_CHECK();
        return UPR_OK;
    });
}

// The status rules the maps entries share, after their own shape check: UPR_E_PARAM for a (illu_dt, e_dt, flags) triple that
// valid_map_dtypes rejects, then UPR_OK (-> *done) for n == 0, then UPR_E_NULL for a missing x, illu, e or result.
inline int maps_check(const MapsArgs& m, int n, bool* done)
{
    *done = true;
    if (!valid_map_dtypes(m.illu_dt, m.e_dt, m.flags)) return UPR_E_PARAM;
    if (n == 0) return UPR_OK;
    if (!m.x || !m.illu || !m.e || (!m.out && !m.out8)) return UPR_E_NULL;
    *done = false;
    return UPR_OK;
}

}  // namespace upr
