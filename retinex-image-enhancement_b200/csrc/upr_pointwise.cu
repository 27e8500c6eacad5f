// upr_pointwise.cu -- the three pointwise epilogues of the classical path (sm_100a).
//
//   a8  Retinex decomposition + recombination   /root/reference/models/model.py:405-413, :442
//         R = x / (illu + eps);  enhanced = R*e + (1 - R)*e^2   (+ its gradient, for training)
//   a5  multi-scale gain + clamp                /root/reference/enhancers/multi_scale.py:97-98
//         out = clamp(enhanced * gain[image], 0, 1)
//   a7  attention gain + clamp                  /root/reference/enhancers/content_aware.py:119-120
//         out = clamp(enhanced * (1 + 0.2*att), 0, 1)
//
// All three are pure HBM streams: one 128-bit load per operand per thread, evict-first
// both ways (nothing is re-read), a persistent grid of 148 x kCtasPerSm CTAs walking the
// frame-major index space.  Every product/sum is an explicitly rounded fp32 operation
// (__fmul_rn/__fadd_rn/__fdiv_rn): torch eager evaluates each Python operator as its own
// kernel, so there is no FMA contraction in the reference and none here -> bit-exact.
#include "upr_maps.cuh"

namespace upr {

constexpr int kPwThreads = 256;
constexpr int kPwCtasPerSm = 8;

// ---- a8 ---------------------------------------------------------------------------------
// plane4 = H*W/4 ; one work item = 4 consecutive pixels of one frame (all three channels).  TI / TE = storage types of illu / e
// (upr_maps.cuh); d = illu + eps is rounded to TI, R and enhanced are f32 (type promotion).
template <typename TI, typename TE, bool kAutocast, bool kWriteRefl, bool kWriteEnh>
__global__ void __launch_bounds__(kPwThreads)
k_recombine_vec(const float* __restrict__ x, const TI* __restrict__ illu, const TE* __restrict__ e,
                float* __restrict__ refl, float* __restrict__ enh, long long plane4, long long items, float eps)
{
    const uint64_t pol = policy_evict_first();
    const long long stride = (long long)gridDim.x * kPwThreads;
    for (long long it = (long long)blockIdx.x * kPwThreads + threadIdx.x; it < items; it += stride) {
        const long long f = it / plane4, p = it - f * plane4;
        const long long o3 = (f * 3 * plane4 + p) * 4, o1 = (f * plane4 + p) * 4;
        const float4 il = MapIO<TI>::ld4(illu + o1, pol);
        const float d[4] = {illu_eps<TI>(il.x, eps), illu_eps<TI>(il.y, eps), illu_eps<TI>(il.z, eps), illu_eps<TI>(il.w, eps)};
        float4 xv[3];
        typename MapIO<TE>::Raw4 ev[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            xv[c] = ld_stream_f4(x + o3 + c * plane4 * 4, pol);
            if (kWriteEnh) ev[c] = MapIO<TE>::ld4raw(e + o3 + c * plane4 * 4, pol);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float4 r, o;
            if (kWriteEnh) {
                const float4 ef = MapIO<TE>::wide4(ev[c]);
                recombine1<TE, kAutocast>(xv[c].x, d[0], ef.x, r.x, o.x);
                recombine1<TE, kAutocast>(xv[c].y, d[1], ef.y, r.y, o.y);
                recombine1<TE, kAutocast>(xv[c].z, d[2], ef.z, r.z, o.z);
                recombine1<TE, kAutocast>(xv[c].w, d[3], ef.w, r.w, o.w);
                st_stream_f4(enh + o3 + c * plane4 * 4, o, pol);
            } else {
                r.x = __fdiv_rn(xv[c].x, d[0]);
                r.y = __fdiv_rn(xv[c].y, d[1]);
                r.z = __fdiv_rn(xv[c].z, d[2]);
                r.w = __fdiv_rn(xv[c].w, d[3]);
            }
            if (kWriteRefl) st_stream_f4(refl + o3 + c * plane4 * 4, r, pol);
        }
    }
}

template <typename TI, typename TE, bool kAutocast, bool kWriteRefl, bool kWriteEnh>
__global__ void __launch_bounds__(kPwThreads)
k_recombine_scalar(const float* __restrict__ x, const TI* __restrict__ illu, const TE* __restrict__ e,
                   float* __restrict__ refl, float* __restrict__ enh, long long plane, long long items, float eps)
{
    const long long stride = (long long)gridDim.x * kPwThreads;
    for (long long it = (long long)blockIdx.x * kPwThreads + threadIdx.x; it < items; it += stride) {
        const long long f = it / plane, p = it - f * plane;
        const float d = illu_eps<TI>(MapIO<TI>::wide(illu[it]), eps);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const long long o = (f * 3 + c) * plane + p;
            float r, v;
            if (kWriteEnh) {
                recombine1<TE, kAutocast>(x[o], d, MapIO<TE>::wide(e[o]), r, v);
                enh[o] = v;
            } else {
                r = __fdiv_rn(x[o], d);
            }
            if (kWriteRefl) refl[o] = r;
        }
    }
}

// ---- a8 gradient --------------------------------------------------------------------------
// What torch autograd computes for the two lines, recomputing d, R and e^2 from the inputs (nothing is saved by the forward).
// gRt, the gradient reaching R, accumulates in the order the autograd engine adds its parts: g_refl (from R's consumers, which
// run first) onto -(gE*c) (rsub), then gE*e (the R*e product, created first, runs last).  The e gradient sums the R*e
// branch, rounded to TE, and the e^2 branch, rounded to TE once (in TE arithmetic without autocast; by the fp32 cast's
// backward under autocast).  The illu gradient is the channel sum of div's "other" gradient in f32 (torch's sum starts from
// 0), then rounded to TI (not at all for the f32 illumination map the network emits under autocast).  grad1 sees the
// illumination side only through d, so it is typed on e's dtype alone.
struct GradPx {
    float gx, ge, gd;
};

template <typename TE, bool kAutocast>
__device__ __forceinline__ GradPx grad1(float x, float d, float e, float gE, float gR, bool has_gE, bool has_gR)
{
    const float r = __fdiv_rn(x, d);
    const float q = __fdiv_rn(r, d);
    float g = gR;
    GradPx o;
    o.ge = 0.0f;
    if (has_gE) {
        const float c = square<TE, kAutocast>(e);
        const float t = -__fmul_rn(gE, c);
        g = __fadd_rn(has_gR ? __fadd_rn(t, gR) : t, __fmul_rn(gE, e));
        float gc = __fmul_rn(gE, __fsub_rn(1.0f, r));
        if (!kAutocast) gc = rnd<TE>(gc);
        const float two_e = kAutocast ? __fmul_rn(2.0f, e) : rnd<TE>(__fmul_rn(2.0f, e));
        o.ge = __fadd_rn(rnd<TE>(__fmul_rn(gE, r)), rnd<TE>(__fmul_rn(gc, two_e)));
    }
    o.gx = __fdiv_rn(g, d);
    o.gd = __fmul_rn(-g, q);
    return o;
}

// Nullable operands: g_enh / g_refl absent = that output got no gradient (g_enh == NULL also when e == NULL, decompose only);
// g_x / g_illu / g_e NULL = that gradient is not wanted.
// (kPwThreads, 1): without a minimum-blocks bound ptxas aims at 64 registers and the f32 instantiation spills 12 bytes around
// the division slow path; it needs 72 (3 CTAs per SM).  The grid stays pw_grid's 148 x 8 CTAs: the later ones start as earlier
// ones finish and keep more loads in flight; a one-wave grid of 148 x 3 measured slower (32x3x640^2: 0.32 -> 0.35 ms f32,
// 0.32 -> 0.37 ms fp16; the same at 16x1080p)
template <typename TI, typename TE, bool kAutocast>
__global__ void __launch_bounds__(kPwThreads, 1)
k_recombine_grad_vec(const float* __restrict__ x, const TI* __restrict__ illu, const TE* __restrict__ e,
                     const float* __restrict__ g_enh, const float* __restrict__ g_refl, float* __restrict__ g_x,
                     TI* __restrict__ g_illu, TE* __restrict__ g_e, long long plane4, long long items, float eps)
{
    const uint64_t pol = policy_evict_first();
    const long long stride = (long long)gridDim.x * kPwThreads;
    const bool has_gE = g_enh != nullptr, has_gR = g_refl != nullptr;
    const float4 zero = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    for (long long it = (long long)blockIdx.x * kPwThreads + threadIdx.x; it < items; it += stride) {
        const long long f = it / plane4, p = it - f * plane4;
        const long long o3 = (f * 3 * plane4 + p) * 4, o1 = (f * plane4 + p) * 4;
        const float4 il = MapIO<TI>::ld4(illu + o1, pol);
        const float d[4] = {illu_eps<TI>(il.x, eps), illu_eps<TI>(il.y, eps), illu_eps<TI>(il.z, eps), illu_eps<TI>(il.w, eps)};
        // one channel at a time: what stays live across the division slow path fits the callee-saved registers (no spills)
        float gd[4];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const long long o = o3 + c * plane4 * 4;
            const float4 xv = ld_stream_f4(x + o, pol);
            const float4 ev = has_gE ? MapIO<TE>::ld4(e + o, pol) : zero;
            const float4 gev = has_gE ? ld_stream_f4(g_enh + o, pol) : zero;
            const float4 grv = has_gR ? ld_stream_f4(g_refl + o, pol) : zero;
            const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, es[4] = {ev.x, ev.y, ev.z, ev.w};
            const float gEs[4] = {gev.x, gev.y, gev.z, gev.w}, gRs[4] = {grv.x, grv.y, grv.z, grv.w};
            float gx[4], ge[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const GradPx g = grad1<TE, kAutocast>(xs[k], d[k], es[k], gEs[k], gRs[k], has_gE, has_gR);
                gx[k] = g.gx;
                ge[k] = g.ge;
                gd[k] = c == 0 ? __fadd_rn(0.0f, g.gd) : __fadd_rn(gd[k], g.gd);
            }
            if (g_x) st_stream_f4(g_x + o, make_float4(gx[0], gx[1], gx[2], gx[3]), pol);
            if (g_e) MapIO<TE>::st4(g_e + o, make_float4(ge[0], ge[1], ge[2], ge[3]), pol);
        }
        if (g_illu) MapIO<TI>::st4(g_illu + o1, make_float4(gd[0], gd[1], gd[2], gd[3]), pol);
    }
}

template <typename TI, typename TE, bool kAutocast>
__global__ void __launch_bounds__(kPwThreads)
k_recombine_grad_scalar(const float* __restrict__ x, const TI* __restrict__ illu, const TE* __restrict__ e,
                        const float* __restrict__ g_enh, const float* __restrict__ g_refl, float* __restrict__ g_x,
                        TI* __restrict__ g_illu, TE* __restrict__ g_e, long long plane, long long items, float eps)
{
    const long long stride = (long long)gridDim.x * kPwThreads;
    const bool has_gE = g_enh != nullptr, has_gR = g_refl != nullptr;
    for (long long it = (long long)blockIdx.x * kPwThreads + threadIdx.x; it < items; it += stride) {
        const long long f = it / plane, p = it - f * plane;
        const float d = illu_eps<TI>(MapIO<TI>::wide(illu[it]), eps);
        float gd = 0.0f;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const long long o = (f * 3 + c) * plane + p;
            const GradPx g = grad1<TE, kAutocast>(x[o], d, has_gE ? MapIO<TE>::wide(e[o]) : 0.0f, has_gE ? g_enh[o] : 0.0f,
                                                  has_gR ? g_refl[o] : 0.0f, has_gE, has_gR);
            gd = __fadd_rn(gd, g.gd);
            if (g_x) g_x[o] = g.gx;
            if (g_e) g_e[o] = MapIO<TE>::narrow(g.ge);
        }
        if (g_illu) g_illu[it] = MapIO<TI>::narrow(gd);
    }
}

// ---- a5 / a7 ----------------------------------------------------------------------------
// kPerPixel == false: gain[f] per frame (a5);  true: gain = 1 + 0.2*att[f][p] per pixel (a7)
// One 128-bit load and one store per trip, all CTAs sweeping the batch linearly inside a ~5 MB window: 6.2-6.3 TB/s on 16 - 192 4K
// frames (a device-to-device copy: 6.5-6.6).  Measured and NOT kept (scripts/dev/clamp_probe.py): 2 / 4 loads in flight per thread
// (window x2 / x4) 5.87 / 5.76 TB/s; a (parts, frame) grid without the index divisions but with every frame open at once 5.70 TB/s
// -- this stream is limited by DRAM page locality, not by bytes in flight or by its 64-bit index arithmetic.
template <bool kPerPixel>
__global__ void __launch_bounds__(kPwThreads)
k_gain_clamp_vec(const float* __restrict__ enh, const float* __restrict__ gain, float* __restrict__ out, int c,
                 long long plane4, long long items)
{
    const uint64_t pol = policy_evict_first();
    const long long stride = (long long)gridDim.x * kPwThreads;
    for (long long it = (long long)blockIdx.x * kPwThreads + threadIdx.x; it < items; it += stride) {
        const long long fc = it / plane4, p = it - fc * plane4;
        const long long f = fc / c;
        const float4 v = ld_stream_f4(enh + it * 4, pol);
        float4 g;
        if (kPerPixel) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(gain + (f * plane4 + p) * 4));
            g.x = __fadd_rn(1.0f, __fmul_rn(0.2f, a.x));
            g.y = __fadd_rn(1.0f, __fmul_rn(0.2f, a.y));
            g.z = __fadd_rn(1.0f, __fmul_rn(0.2f, a.z));
            g.w = __fadd_rn(1.0f, __fmul_rn(0.2f, a.w));
        } else {
            const float s = __ldg(gain + f);
            g = make_float4(s, s, s, s);
        }
        float4 o;
        o.x = clamp01_keep_nan(__fmul_rn(v.x, g.x));
        o.y = clamp01_keep_nan(__fmul_rn(v.y, g.y));
        o.z = clamp01_keep_nan(__fmul_rn(v.z, g.z));
        o.w = clamp01_keep_nan(__fmul_rn(v.w, g.w));
        st_stream_f4(out + it * 4, o, pol);
    }
}

template <bool kPerPixel>
__global__ void __launch_bounds__(kPwThreads)
k_gain_clamp_scalar(const float* __restrict__ enh, const float* __restrict__ gain, float* __restrict__ out, int c,
                    long long plane, long long items)
{
    const long long stride = (long long)gridDim.x * kPwThreads;
    for (long long it = (long long)blockIdx.x * kPwThreads + threadIdx.x; it < items; it += stride) {
        const long long fc = it / plane, p = it - fc * plane;
        const long long f = fc / c;
        const float g = kPerPixel ? __fadd_rn(1.0f, __fmul_rn(0.2f, gain[f * plane + p])) : gain[f];
        out[it] = clamp01_keep_nan(__fmul_rn(enh[it], g));
    }
}

static inline int pw_grid(long long items)
{
    const long long want = (items + kPwThreads - 1) / kPwThreads;
    return int(std::max<long long>(1, std::min<long long>(want, (long long)kNumSMsB200 * kPwCtasPerSm)));
}

template <typename TI, typename TE, bool AC, bool R, bool E>
static int recombine_launch(const float* x, const TI* illu, const TE* e, float* refl, float* enh, int n, int h, int w,
                            float eps, cudaStream_t s)
{
    const long long plane = (long long)h * w;
    const bool vec = plane % 4 == 0 && aligned16(x) && aligned4px(illu) && (!E || (aligned4px(e) && aligned16(enh))) &&
                     (!R || aligned16(refl));
    if (vec) {
        const long long items = (long long)n * (plane / 4);
        k_recombine_vec<TI, TE, AC, R, E><<<pw_grid(items), kPwThreads, 0, s>>>(x, illu, e, refl, enh, plane / 4, items, eps);
    } else {
        const long long items = (long long)n * plane;
        k_recombine_scalar<TI, TE, AC, R, E><<<pw_grid(items), kPwThreads, 0, s>>>(x, illu, e, refl, enh, plane, items, eps);
    }
    UPR_LAUNCH_CHECK();
    return UPR_OK;
}

// upr_retinex_recombine_maps / _typed on map types (TI, TE); the arguments are checked (refl or enh is given; enh only with e).
// Without e, or without enh, only R is formed, and e's dtype and the flag are moot.
template <typename TI, typename TE, bool AC>
static int recombine_maps(const float* x, const void* illu_v, const void* e_v, float* refl, float* enh, int n, int h,
                          int w, float eps, cudaStream_t s)
{
    const TI* illu = static_cast<const TI*>(illu_v);
    const TE* e = static_cast<const TE*>(e_v);
    if (!e || !enh)
        return recombine_launch<TI, TI, false, true, false>(x, illu, nullptr, refl, nullptr, n, h, w, eps, s);
    return refl ? recombine_launch<TI, TE, AC, true, true>(x, illu, e, refl, enh, n, h, w, eps, s)
                : recombine_launch<TI, TE, AC, false, true>(x, illu, e, nullptr, enh, n, h, w, eps, s);
}

// the checked arguments of upr_retinex_recombine_maps / _typed, dispatched on (illu dtype, e dtype, autocast)
static int recombine_typed(const float* x, const void* illu, int illu_dt, const void* e, int e_dt, int flags, float* refl,
                           float* enh, int n, int h, int w, float eps, cudaStream_t s)
{
    return with_map_types(illu_dt, e_dt, flags, [&](auto ti, auto te, auto ac) {
        return recombine_maps<typename decltype(ti)::type, typename decltype(te)::type, decltype(ac)::value>(x, illu, e, refl, enh,
                                                                                                              n, h, w, eps, s);
    });
}

// upr_retinex_recombine_grad_typed on map types (TI, TE), arguments checked.  The vector kernel needs every map operand
// aligned to 4 pixels of its own dtype (aligned4px), as the forward does.
template <typename TI, typename TE, bool AC>
static int recombine_grad(const float* x, const void* illu_v, const void* e_v, const float* g_enh, const float* g_refl,
                          float* g_x, void* g_illu_v, void* g_e_v, int n, int h, int w, float eps, cudaStream_t s)
{
    const TI* illu = static_cast<const TI*>(illu_v);
    const TE* e = static_cast<const TE*>(e_v);
    TI* g_illu = static_cast<TI*>(g_illu_v);
    TE* g_e = static_cast<TE*>(g_e_v);
    const long long plane = (long long)h * w;
    const bool vec = plane % 4 == 0 && aligned16(x) && aligned4px(illu) && (!e || aligned4px(e)) &&
                     (!g_enh || aligned16(g_enh)) && (!g_refl || aligned16(g_refl)) && (!g_x || aligned16(g_x)) &&
                     (!g_illu || aligned4px(g_illu)) && (!g_e || aligned4px(g_e));
    if (vec) {
        const long long items = (long long)n * (plane / 4);
        k_recombine_grad_vec<TI, TE, AC><<<pw_grid(items), kPwThreads, 0, s>>>(x, illu, e, g_enh, g_refl, g_x, g_illu, g_e,
                                                                              plane / 4, items, eps);
    } else {
        const long long items = (long long)n * plane;
        k_recombine_grad_scalar<TI, TE, AC><<<pw_grid(items), kPwThreads, 0, s>>>(x, illu, e, g_enh, g_refl, g_x, g_illu,
                                                                                 g_e, plane, items, eps);
    }
    UPR_LAUNCH_CHECK();
    return UPR_OK;
}

template <bool P>
static int gain_launch(const float* enh, const float* gain, float* out, int n, int c, int h, int w, cudaStream_t s)
{
    const long long plane = (long long)h * w;
    const bool vec = plane % 4 == 0 && aligned16(enh) && aligned16(out) && (!P || aligned16(gain));
    if (vec) {
        const long long items = (long long)n * c * (plane / 4);
        k_gain_clamp_vec<P><<<pw_grid(items), kPwThreads, 0, s>>>(enh, gain, out, c, plane / 4, items);
    } else {
        const long long items = (long long)n * c * plane;
        k_gain_clamp_scalar<P><<<pw_grid(items), kPwThreads, 0, s>>>(enh, gain, out, c, plane, items);
    }
    UPR_LAUNCH_CHECK();
    return UPR_OK;
}

int scale_clamp_launch(const float* enh, const float* gain, float* out, int n, int c, int h, int w, cudaStream_t s)
{
    return gain_launch<false>(enh, gain, out, n, c, h, w, s);
}

// ---- save_image quantiser (enhancers/simple_enhance.py:65-100) -----------------------------------
// [n][c][h][w] f32 -> [n][h][w][c] u8 with save_u8 (upr_common.cuh).  c = 1 (illumination maps) or 3 (frames).  One thread
// per 4 pixels: c 128-bit loads, 4c contiguous bytes stored.
template <int C>
__global__ void __launch_bounds__(kPwThreads)
k_quantize_u8(const float* __restrict__ x, unsigned char* __restrict__ out, long long plane, long long items)
{
    const long long plane4 = plane / 4;
    const long long stride = (long long)gridDim.x * kPwThreads;
    for (long long it = (long long)blockIdx.x * kPwThreads + threadIdx.x; it < items; it += stride) {
        const long long f = it / plane4, p = it - f * plane4;
        unsigned q[C][4];
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float4 v = __ldcs(reinterpret_cast<const float4*>(x + (f * C + c) * plane) + p);
            const float a[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) q[c][k] = save_u8(a[k]);
        }
        unsigned char* o = out + (f * plane + p * 4) * C;
        if constexpr (C == 1) *reinterpret_cast<unsigned*>(o) = pack4_u8(q[0]);
        else st_rgb4_u8(o, q);
    }
}

template <int C>
__global__ void __launch_bounds__(kPwThreads)
k_quantize_u8_scalar(const float* __restrict__ x, unsigned char* __restrict__ out, long long plane, long long items)
{
    const long long stride = (long long)gridDim.x * kPwThreads;
    for (long long it = (long long)blockIdx.x * kPwThreads + threadIdx.x; it < items; it += stride) {
        const long long f = it / plane, p = it - f * plane;
#pragma unroll
        for (int c = 0; c < C; ++c)
            out[it * C + c] = (unsigned char)save_u8(x[(f * C + c) * plane + p]);
    }
}

}  // namespace upr

extern "C" {

int upr_quantize_u8_f32(const float* x_nchw, unsigned char* out_nhwc, int n, int c, int h, int w, upr_stream_t stream)
{
    if (n < 0 || h <= 0 || w <= 0 || (c != 1 && c != 3)) return UPR_E_SHAPE;
    if (n == 0) return UPR_OK;
    if (!x_nchw || !out_nhwc) return UPR_E_NULL;
    auto s = static_cast<cudaStream_t>(stream);
    const long long plane = (long long)h * w;
    if (plane % 4 == 0 && upr::aligned16(x_nchw) && (reinterpret_cast<uintptr_t>(out_nhwc) & 3u) == 0) {
        const long long items = (long long)n * (plane / 4);
        if (c == 1) upr::k_quantize_u8<1><<<upr::pw_grid(items), upr::kPwThreads, 0, s>>>(x_nchw, out_nhwc, plane, items);
        else upr::k_quantize_u8<3><<<upr::pw_grid(items), upr::kPwThreads, 0, s>>>(x_nchw, out_nhwc, plane, items);
    } else {
        const long long items = (long long)n * plane;
        if (c == 1) upr::k_quantize_u8_scalar<1><<<upr::pw_grid(items), upr::kPwThreads, 0, s>>>(x_nchw, out_nhwc, plane, items);
        else upr::k_quantize_u8_scalar<3><<<upr::pw_grid(items), upr::kPwThreads, 0, s>>>(x_nchw, out_nhwc, plane, items);
    }
    UPR_LAUNCH_CHECK();
    return UPR_OK;
}

int upr_retinex_quantize_typed_u8(const float* x_nchw, const void* illu_n1hw, int illu_dtype, const void* e_nchw, int e_dtype,
                                  int flags, unsigned char* enh_nhwc, unsigned char* illu_nhw1, int n, int h, int w, float eps,
                                  upr_stream_t stream)
{
    if (n < 0 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    const upr::MapsArgs m{x_nchw, illu_n1hw, illu_dtype, e_nchw, e_dtype, flags, eps, nullptr, enh_nhwc, illu_nhw1};
    bool done;
    const int rc = upr::maps_check(m, n, &done);
    if (done) return rc;
    return upr::maps_epilogue(m, n, h, w, upr::NoGain{}, static_cast<cudaStream_t>(stream));
}

int upr_retinex_recombine_f32(const float* x, const float* illu, const float* e, float* refl, float* enh, int n, int h,
                              int w, float eps, upr_stream_t stream)
{
    if (n < 0 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    if (n == 0) return UPR_OK;
    if (!x || !illu || !e || !enh) return UPR_E_NULL;
    auto s = static_cast<cudaStream_t>(stream);
    return refl ? upr::recombine_launch<float, float, false, true, true>(x, illu, e, refl, enh, n, h, w, eps, s)
                : upr::recombine_launch<float, float, false, false, true>(x, illu, e, nullptr, enh, n, h, w, eps, s);
}

int upr_retinex_decompose_f32(const float* x, const float* illu, float* refl, int n, int h, int w, float eps,
                              upr_stream_t stream)
{
    if (n < 0 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    if (n == 0) return UPR_OK;
    if (!x || !illu || !refl) return UPR_E_NULL;
    return upr::recombine_launch<float, float, false, true, false>(x, illu, nullptr, refl, nullptr, n, h, w, eps,
                                                                   static_cast<cudaStream_t>(stream));
}

int upr_retinex_recombine_maps(const float* x, const void* illu, const void* e, int map_dtype, int flags, float* refl,
                               float* enh, int n, int h, int w, float eps, upr_stream_t stream)
{
    if (n < 0 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    if (map_dtype < UPR_DT_F32 || map_dtype > UPR_DT_BF16 || (flags & ~UPR_RETINEX_AUTOCAST)) return UPR_E_PARAM;
    if (n == 0) return UPR_OK;
    if (!x || !illu || (!refl && !enh) || (!e && enh)) return UPR_E_NULL;
    return upr::recombine_typed(x, illu, map_dtype, e, map_dtype, flags, refl, enh, n, h, w, eps, static_cast<cudaStream_t>(stream));
}

int upr_retinex_recombine_typed(const float* x, const void* illu, int illu_dtype, const void* e, int e_dtype, int flags,
                                float* refl, float* enh, int n, int h, int w, float eps, upr_stream_t stream)
{
    if (n < 0 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    if (!upr::valid_map_dtypes(illu_dtype, e_dtype, flags)) return UPR_E_PARAM;
    if (n == 0) return UPR_OK;
    if (!x || !illu || (!refl && !enh) || (!e && enh)) return UPR_E_NULL;
    return upr::recombine_typed(x, illu, illu_dtype, e, e_dtype, flags, refl, enh, n, h, w, eps, static_cast<cudaStream_t>(stream));
}

int upr_retinex_recombine_grad_typed(const float* x, const void* illu, int illu_dtype, const void* e, int e_dtype, int flags,
                                     const float* g_enh, const float* g_refl, float* g_x, void* g_illu, void* g_e, int n, int h,
                                     int w, float eps, upr_stream_t stream)
{
    if (n < 0 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    if (!upr::valid_map_dtypes(illu_dtype, e_dtype, flags)) return UPR_E_PARAM;
    if (n == 0) return UPR_OK;
    if (!x || !illu || (!g_enh && !g_refl) || (!e && (g_enh || g_e))) return UPR_E_NULL;
    if (!g_x && !g_illu && !g_e) return UPR_OK;
    auto s = static_cast<cudaStream_t>(stream);
    return upr::with_map_types(illu_dtype, e_dtype, flags, [&](auto ti, auto te, auto ac) {
        return upr::recombine_grad<typename decltype(ti)::type, typename decltype(te)::type, decltype(ac)::value>(
            x, illu, e, g_enh, g_refl, g_x, g_illu, g_e, n, h, w, eps, s);
    });
}

int upr_retinex_recombine_grad(const float* x, const void* illu, const void* e, int map_dtype, int flags,
                               const float* g_enh, const float* g_refl, float* g_x, void* g_illu, void* g_e, int n, int h,
                               int w, float eps, upr_stream_t stream)
{
    return upr_retinex_recombine_grad_typed(x, illu, map_dtype, e, map_dtype, flags, g_enh, g_refl, g_x, g_illu, g_e, n, h, w,
                                            eps, stream);
}

int upr_scale_clamp_f32(const float* enh, const float* gain_per_image, float* out, int n, int c, int h, int w,
                        upr_stream_t stream)
{
    if (n < 0 || c <= 0 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    if (n == 0) return UPR_OK;
    if (!enh || !gain_per_image || !out) return UPR_E_NULL;
    return upr::gain_launch<false>(enh, gain_per_image, out, n, c, h, w, static_cast<cudaStream_t>(stream));
}

int upr_attention_apply_f32(const float* enh, const float* att, float* out, int n, int c, int h, int w,
                            upr_stream_t stream)
{
    if (n < 0 || c <= 0 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    if (n == 0) return UPR_OK;
    if (!enh || !att || !out) return UPR_E_NULL;
    return upr::gain_launch<true>(enh, att, out, n, c, h, w, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
