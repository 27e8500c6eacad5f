// upr_saliency.cu -- content-aware saliency and attention maps (sm_100a).
//
// Replaces ContentAwareEnhancer.compute_saliency_map / compute_attention_map
// (/root/reference/enhancers/content_aware.py:19-59, :61-91):
//   gray = BGR2GRAY(u8 quantise(x))                     OpenCV fixed point (SURVEY Appendix A.4)
//   lap  = |cv2.Laplacian(gray, CV_64F)|                4-neighbour, BORDER_REFLECT_101 (integers <= 1020)
//   blur = cv2.GaussianBlur(lap, (15,15), 0)            sigma 2.6, separable, fp64, BORDER_REFLECT_101
//   sal  = float32((blur - min) / (max - min + 1e-8))   per image
//   att  = sal * (1 / (luma(x) + 0.1)); att = (att - min) / (max - min + 1e-8)   fp32, per image
//
// K5 k_saliency_stream: one warp per (frame, 256-column band, row segment).  The reflect-101 extension commutes with
//    the (mirror symmetric) Laplacian and Gaussian, so the whole chain is evaluated on the reflected plane: gray (exact
//    integers in fp32) -> |lap| -> fp16 ring of 16 rows -> vertical then horizontal 15-tap pass in fp32 -> un-normalised
//    blur stored as fp32, per-warp min/max folded into per-image ordered-integer atomics (exact, order independent).
// K6 k_attention_raw: sal normalise + luma division fused, fp32 min/max of the raw attention per image.
// K7 k_normalize: (v - min) / (max - min + 1e-8) in place (used for both maps).
#include <algorithm>
#include <cmath>
#include <mutex>

#include <cuda_fp16.h>

#include "upr_maps.cuh"

namespace upr {

constexpr int kSalThreads = 256;

__device__ __forceinline__ int reflect101_s(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * (len - 1) - p;
    return p;
}

// order-preserving map double <-> unsigned 64 (for exact atomic min/max)
__device__ __forceinline__ unsigned long long dbl_key(double v)
{
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_dbl(unsigned long long k)
{
    const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}
__device__ __forceinline__ unsigned flt_key(float v)
{
    const unsigned b = __float_as_uint(v);
    return (b >> 31) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_flt(unsigned k)
{
    const unsigned b = (k >> 31) ? (k & 0x7fffffffu) : ~k;
    return __uint_as_float(b);
}

struct SalMinMax {           // per image, 32 bytes
    unsigned long long blur_min, blur_max;   // ordered keys of fp64 values
    unsigned att_min, att_max;               // ordered keys of fp32 values
    unsigned pad0, pad1;
};

__global__ void k_sal_reset(SalMinMax* mm, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    mm[i].blur_min = ~0ull; mm[i].blur_max = 0ull;
    mm[i].att_min = ~0u; mm[i].att_max = 0u;
    mm[i].pad0 = mm[i].pad1 = 0;
}

// ---------------------------------------------------------------------------------------------
// K5 k_saliency_stream: a row-streaming, one-warp-per-CTA kernel.
//   (A 64x64 shared-memory tile kernel with an fp64 blur executed 271 SASS instructions per pixel -- 56 % halo
//   re-computation of the gray stage (80x80 per 64x64), scalar reflect-indexed loads, 15 shared loads per output and
//   pass, an fp64 FMA chain: 1.76 ms against 0.65 ms on 16 x 4K, profiles/r2_content_aware_full.md.)  A warp owns a band of 256 columns (lane = 8 columns; lanes 0 and 31 are the +-8 halo, 240 columns
//   are written) and marches down a row segment:
//     load row k (two 128-bit loads per plane and lane) -> quantise/gray on the FMA pipe (exact integer arithmetic in
//     fp32, see upr_clahe.cu) -> |lap| of row k-1 (vertical neighbours from registers, the two horizontal ones by
//     shuffle) -> fp16 ring of the last 16 |lap| rows in shared memory (integers <= 1020, and their pair sums <= 2040,
//     are exact in fp16; the ring is private per lane and column, so it needs no synchronisation) -> VERTICAL 15-tap
//     pass of row k-8 (symmetric taps paired) -> one fp32 row exchanged through a per-warp buffer (__syncwarp only) ->
//     HORIZONTAL pass -> un-normalised blur (fp32) + running min/max.
//   Vertical-then-horizontal and fp32 accumulation differ from OpenCV's fp64 rows-then-columns by ~2e-7 relative --
//   the same order as the fp32 rounding of the stored blur itself, and far inside the stated 1e-4 bound (SURVEY 8c).
//   Row segments overlap by 16 rows, bands by 16 columns (amplification ~1.07 x 1.06 instead of 1.56).
// ---------------------------------------------------------------------------------------------
constexpr int kSsLaneCols = 8;
constexpr int kSsBandCols = 30 * kSsLaneCols;      // 240 written columns per warp
constexpr int kSsRingRows = 16;                    // power of two: slot offsets wrap with a mask
constexpr int kSsRingRowBytes = 32 * kSsLaneCols * 2;   // 512
constexpr int kSsRingBytes = kSsRingRows * kSsRingRowBytes;   // 8192

struct GaussTapsF {
    float t[8];
};

__device__ __forceinline__ void ss_load8(const float* __restrict__ row, int c0, int w, bool vec, float v[8])
{
    if (vec) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(row + c0));
        const float4 b = __ldg(reinterpret_cast<const float4*>(row + c0 + 4));
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = __ldg(row + reflect101_s(c0 + i, w));
    }
}

__global__ void __launch_bounds__(32)
k_saliency_stream(const float* __restrict__ x, int h, int w, int bands, int seg_rows, float* __restrict__ blur_out,
                  SalMinMax* __restrict__ mm, const GaussTapsF taps)
{
    __shared__ __align__(16) unsigned char s_ring[kSsRingBytes];
    __shared__ __align__(16) float s_row[2][2 * 34 * 4];

    const int lane = threadIdx.x;
    const int band = blockIdx.x % bands, seg = blockIdx.x / bands;
    const int f = blockIdx.y;
    const int r0 = seg * seg_rows, r1 = min(r0 + seg_rows, h);
    if (r0 >= h) return;
    const int c0 = band * kSsBandCols - kSsLaneCols + lane * kSsLaneCols;   // plane column of this lane's first pixel
    const long long plane = (long long)h * w;
    const float* img = x + (long long)f * 3 * plane;
    const bool vec = (w % 4 == 0) && c0 >= 0 && c0 + kSsLaneCols <= w && aligned16(x);
    const bool writer = lane >= 1 && lane <= 30 && c0 < w;
    const bool vec_out = vec && aligned16(blur_out);

    const uint32_t ring_lane = uint32_t(__cvta_generic_to_shared(s_ring)) + uint32_t(lane) * 16u;
    float g0[8], g1[8], g2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) g0[i] = g1[i] = g2[i] = 0.0f;
    float mn = INFINITY, mx = -INFINITY;
    uint32_t slot = 0;   // byte offset of the ring row that receives the next |lap| row

    float nr[8], ng[8], nb[8];
    auto load_row = [&](int k) {
        const float* rowp = img + (long long)reflect101_s(k, h) * w;
        ss_load8(rowp, c0, w, vec, nr);
        ss_load8(rowp + plane, c0, w, vec, ng);
        ss_load8(rowp + 2 * plane, c0, w, vec, nb);
    };
    load_row(r0 - 8);
    for (int k = r0 - 8; k < r1 + 8; ++k) {
        // ---- gray(k) ----
        {
            // software pipeline: row k+1 is requested before row k is converted
            float r[8], g[8], b[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) { r[i] = nr[i]; g[i] = ng[i]; b[i] = nb[i]; }
            if (k + 1 < r1 + 8) load_row(k + 1);
            // L2 prefetch two rows ahead (row k+1 is already in registers).  Swept on 16 x 4K, saliency op: none 0.923 ms, 2 rows
            // 0.847, 3 rows 0.850, 4 rows 0.859, 6 rows 0.904, 8 rows 0.967, 12 rows 1.025
            if (vec && k + 2 < r1 + 8) {
                const float* rp = img + (long long)reflect101_s(k + 2, h) * w + c0;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(rp));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + plane));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + 2 * plane));
            }
            uint32_t m = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) m = __vimax3_u32(m, __float_as_uint(r[i]), __vimax3_u32(__float_as_uint(g[i]), __float_as_uint(b[i]), 0u));
            if (m <= 0x3F800000u) {   // all in [+0, 1]: trunc(v*255) == RZ(v*255 + 2^23) - 2^23
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float qr = __fsub_rn(__fadd_rz(__fmul_rn(r[i], 255.0f), 8388608.0f), 8388608.0f);
                    const float qg = __fsub_rn(__fadd_rz(__fmul_rn(g[i], 255.0f), 8388608.0f), 8388608.0f);
                    const float qb = __fsub_rn(__fadd_rz(__fmul_rn(b[i], 255.0f), 8388608.0f), 8388608.0f);
                    // (9798 R + 19235 G + 3735 B + 16384) >> 15: every partial sum is an integer < 2^24
                    const float sgr = __fmaf_rn(qb, 3735.0f, __fmaf_rn(qg, 19235.0f, __fmaf_rn(qr, 9798.0f, 16384.0f)));
                    g2[i] = __fsub_rn(__fmaf_rz(sgr, 0.000030517578125f, 8388608.0f), 8388608.0f);
                }
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    g2[i] = float((quantize_u8(r[i]) * 9798 + quantize_u8(g[i]) * 19235 + quantize_u8(b[i]) * 3735 + 16384) >> 15);
            }
        }
        // ---- |lap|(k-1) -> ring ----
        if (k >= r0 - 6) {
            const float left = __shfl_up_sync(0xffffffffu, g1[7], 1), right = __shfl_down_sync(0xffffffffu, g1[0], 1);
            float a[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float l = i == 0 ? left : g1[i - 1], rr = i == 7 ? right : g1[i + 1];
                a[i] = fabsf(__fmaf_rn(g1[i], -4.0f, __fadd_rn(__fadd_rn(g0[i], g2[i]), __fadd_rn(l, rr))));
            }
            const __half2 h01 = __floats2half2_rn(a[0], a[1]), h23 = __floats2half2_rn(a[2], a[3]);
            const __half2 h45 = __floats2half2_rn(a[4], a[5]), h67 = __floats2half2_rn(a[6], a[7]);
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(ring_lane + slot), "r"(*reinterpret_cast<const uint32_t*>(&h01)),
                         "r"(*reinterpret_cast<const uint32_t*>(&h23)), "r"(*reinterpret_cast<const uint32_t*>(&h45)),
                         "r"(*reinterpret_cast<const uint32_t*>(&h67)) : "memory");
            // ---- vertical pass of row k-8, horizontal pass, output ----
            if (k >= r0 + 8) {
                // rows k-1-i live at (slot - i*512) & 8191; centre i = 7
                auto ring_row = [&](int i, __half2 v[4]) {
                    const uint32_t a4 = ring_lane + ((slot - uint32_t(i) * kSsRingRowBytes) & uint32_t(kSsRingBytes - 1));
                    uint32_t u0, u1, u2, u3;
                    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(u0), "=r"(u1), "=r"(u2), "=r"(u3) : "r"(a4));
                    v[0] = *reinterpret_cast<__half2*>(&u0); v[1] = *reinterpret_cast<__half2*>(&u1);
                    v[2] = *reinterpret_cast<__half2*>(&u2); v[3] = *reinterpret_cast<__half2*>(&u3);
                };
                float vsum[8];
                {
                    __half2 c[4];
                    ring_row(7, c);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float2 cf = __half22float2(c[j]);
                        vsum[2 * j] = __fmul_rn(taps.t[0], cf.x);
                        vsum[2 * j + 1] = __fmul_rn(taps.t[0], cf.y);
                    }
                }
#pragma unroll
                for (int d = 1; d <= 7; ++d) {
                    __half2 p[4], q[4];
                    ring_row(7 - d, p);
                    ring_row(7 + d, q);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float2 sf = __half22float2(__hadd2(p[j], q[j]));   // integers <= 2040: exact in fp16
                        vsum[2 * j] = __fmaf_rn(taps.t[d], sf.x, vsum[2 * j]);
                        vsum[2 * j + 1] = __fmaf_rn(taps.t[d], sf.y, vsum[2 * j + 1]);
                    }
                }
                // exchange buffer: first halves (columns 0..3) of all lanes, then second halves -- every 128-bit access of
                // the warp is contiguous (an interleaved [lane][8] layout costs 8 wavefronts per access instead of 4)
                float4* rowA = reinterpret_cast<float4*>(s_row[k & 1]) + 1;      // slot -1 and slot 32 are padding
                float4* rowB = rowA + 34;
                rowA[lane] = make_float4(vsum[0], vsum[1], vsum[2], vsum[3]);
                rowB[lane] = make_float4(vsum[4], vsum[5], vsum[6], vsum[7]);
                __syncwarp();
                float bwin[24];
                {
                    const float4 t0 = rowA[lane - 1], t1 = rowB[lane - 1], t4 = rowA[lane + 1], t5 = rowB[lane + 1];
                    bwin[0] = t0.x; bwin[1] = t0.y; bwin[2] = t0.z; bwin[3] = t0.w;
                    bwin[4] = t1.x; bwin[5] = t1.y; bwin[6] = t1.z; bwin[7] = t1.w;
#pragma unroll
                    for (int i = 0; i < 8; ++i) bwin[8 + i] = vsum[i];
                    bwin[16] = t4.x; bwin[17] = t4.y; bwin[18] = t4.z; bwin[19] = t4.w;
                    bwin[20] = t5.x; bwin[21] = t5.y; bwin[22] = t5.z; bwin[23] = t5.w;
                }
                float o[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float acc = __fmul_rn(taps.t[0], bwin[8 + i]);
#pragma unroll
                    for (int d = 1; d <= 7; ++d) acc = __fmaf_rn(taps.t[d], __fadd_rn(bwin[8 + i - d], bwin[8 + i + d]), acc);
                    o[i] = acc;
                }
                const int m = k - 8;   // output row
                if (writer) {
                    float* dst = blur_out + (long long)f * plane + (long long)m * w + c0;
                    if (vec_out) {
                        __stcg(reinterpret_cast<float4*>(dst), make_float4(o[0], o[1], o[2], o[3]));
                        __stcg(reinterpret_cast<float4*>(dst + 4), make_float4(o[4], o[5], o[6], o[7]));
#pragma unroll
                        for (int i = 0; i < 8; ++i) { mn = fminf(mn, o[i]); mx = fmaxf(mx, o[i]); }
                    } else {
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            if (c0 + i >= 0 && c0 + i < w) { dst[i] = o[i]; mn = fminf(mn, o[i]); mx = fmaxf(mx, o[i]); }
                    }
                }
            }
            slot = (slot + kSsRingRowBytes) & uint32_t(kSsRingBytes - 1);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) { g0[i] = g1[i]; g1[i] = g2[i]; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0 && mn <= mx) {
        atomicMin(&mm[f].blur_min, dbl_key(double(mn)));
        atomicMax(&mm[f].blur_max, dbl_key(double(mx)));
    }
}

// ---------------------------------------------------------------------------------------------
// K5 second generation, k_saliency_stream2.  ncu on k_saliency_stream: 102 executed instructions per pixel at 114 registers,
// issue-bound (0.65 ms per 16 x 4K for 16 B/px); tighter launch bounds only add spills (18 -> 32 warps/SM: 0.89 -> 1.13 ms,
// profiles/r4_saliency.md).  So the instruction stream itself is cut:
//   * TWO output rows per iteration.  The vertical pass streams the 16 live |lap| rows through registers once and feeds both
//     rows' accumulators (half the shared-memory loads per pixel); no symmetric pairing -- a pair add plus an FMA costs the same
//     two issue slots as two FMAs;
//   * packed fp32 arithmetic (Blackwell FFMA2 / FADD2 / FMUL2: two fp32 lanes per issue slot) on natural column pairs -- the
//     registers a 128-bit load delivers -- for quantisation, gray, the vertical part of the Laplacian, the whole vertical pass
//     and the FMA half of the horizontal pass (its pair sums are scalar adds that land in aligned register pairs);
//   * the |lap| ring stays fp16 (exact) and every ring row is converted ONCE per iteration for both output rows; the two rows
//     formed in the iteration itself never leave registers.  (An fp32 ring needs no conversions but twice the shared-memory
//     wavefronts: ncu had that variant at 84 % of the L1/shared data pipe with 44 % of the issue slots used.)
// Same arithmetic as the first generation up to the order of the fp32 tap sums (still far inside the 1e-4 bound, tests).
// ---------------------------------------------------------------------------------------------
constexpr int kS2RingRowBytes = 512;                  // 32 lanes x 8 columns x fp16 (integers <= 1020: exact)
constexpr int kS2RingBytes = 16 * kS2RingRowBytes;    // 16 live |lap| rows
constexpr int kS2XRowFloats = 2 * 34 * 4;
constexpr int kS2SegRows = 64;                        // rows per warp (+ 16 halo rows)             // one exchanged row: [half][34 lane slots] float4 (slots -1 and 32 are padding)

// gray of 8 pixels from planar f32 rows, packed column pairs.  kFast: every value is in [+0, 1] (see k_saliency_stream).
__device__ __forceinline__ void s2_gray8(const float (&r)[8], const float (&g)[8], const float (&b)[8], f32x2 (&out)[4])
{
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) m = __vimax3_u32(m, __float_as_uint(r[i]), __vimax3_u32(__float_as_uint(g[i]), __float_as_uint(b[i]), 0u));
    if (m <= 0x3F800000u) {
        const f32x2 k255 = pk2(255.0f, 255.0f), kmagic = pk2(8388608.0f, 8388608.0f);
        const f32x2 kr = pk2(9798.0f, 9798.0f), kg = pk2(19235.0f, 19235.0f), kb = pk2(3735.0f, 3735.0f);
        const f32x2 khalf = pk2(16384.0f, 16384.0f), kinv = pk2(0.000030517578125f, 0.000030517578125f);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            // trunc(v * 255) == RZ(RN(v * 255) + 2^23) - 2^23; the dot product and the shift are exact integer arithmetic in fp32
            const f32x2 qr = sub2(add2_rz(mul2(pk2(r[2 * j], r[2 * j + 1]), k255), kmagic), kmagic);
            const f32x2 qg = sub2(add2_rz(mul2(pk2(g[2 * j], g[2 * j + 1]), k255), kmagic), kmagic);
            const f32x2 qb = sub2(add2_rz(mul2(pk2(b[2 * j], b[2 * j + 1]), k255), kmagic), kmagic);
            const f32x2 sgr = fma2(qb, kb, fma2(qg, kg, fma2(qr, kr, khalf)));
            out[j] = sub2(fma2_rz(sgr, kinv, kmagic), kmagic);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float a = float((quantize_u8(r[2 * j]) * 9798 + quantize_u8(g[2 * j]) * 19235 + quantize_u8(b[2 * j]) * 3735 + 16384) >> 15);
            const float c = float((quantize_u8(r[2 * j + 1]) * 9798 + quantize_u8(g[2 * j + 1]) * 19235 + quantize_u8(b[2 * j + 1]) * 3735 + 16384) >> 15);
            out[j] = pk2(a, c);
        }
    }
}

// |4-neighbour Laplacian| of the middle row, 8 columns: vertical part packed, horizontal neighbours scalar (lane edges by shuffle)
__device__ __forceinline__ void s2_lap8(const f32x2 (&up)[4], const f32x2 (&mid)[4], const f32x2 (&dn)[4], float (&out)[8])
{
    const f32x2 kneg4 = pk2(-4.0f, -4.0f);
    float m[8], v[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        upk2(mid[j], m[2 * j], m[2 * j + 1]);
        upk2(fma2(mid[j], kneg4, add2(up[j], dn[j])), v[2 * j], v[2 * j + 1]);
    }
    const float left = __shfl_up_sync(0xffffffffu, m[7], 1), right = __shfl_down_sync(0xffffffffu, m[0], 1);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float l = i == 0 ? left : m[i - 1], rr = i == 7 ? right : m[i + 1];
        out[i] = fabsf(__fadd_rn(v[i], __fadd_rn(l, rr)));
    }
}

// Requires w % 8 == 0, w >= 16, h >= 16 and 16-byte aligned planes (the named shapes); k_saliency_stream serves everything else.  There is
// no scalar or reflect-indexed code in this kernel (its instruction stream must stay inside the instruction cache): every lane loads
// aligned vectors from a clamped column, rows reflect with one comparison, and the two halo lanes that hang over the left / right
// image border take their gray values -- the reflection of columns 1..8 resp. w-2..w-9 -- from the neighbouring lanes by shuffle.
// kLum: also leaves luma(x) = .299 r + .587 g + .114 b (content_aware.py:76-78, separately rounded like torch) of the segment's own
// rows in `lum_out` (frame stride lum_stride floats), so that the attention pass reads 4 instead of 12 B/px.
template <bool kLum>
__global__ void __launch_bounds__(32, 12)
k_saliency_stream2(const float* __restrict__ x, int h, int w, int bands, int seg_rows, float* __restrict__ blur_out,
                   SalMinMax* __restrict__ mm, const GaussTapsF taps, float* __restrict__ lum_out, long long lum_stride)
{
    __shared__ __align__(16) unsigned char s_ring[kS2RingBytes];
    __shared__ __align__(16) float s_xch[2][2][kS2XRowFloats];   // [iteration parity][row m / m+1]

    const int lane = threadIdx.x;
    const int band = blockIdx.x % bands, seg = blockIdx.x / bands;
    const int f = blockIdx.y;
    const int r0 = seg * seg_rows, r1 = min(r0 + seg_rows, h);
    if (r0 >= h) return;
    // Odd segments walk UP from their last row: neighbouring segments then start from a common boundary row at the same time and
    // arrive at the other boundary together, so the 8 warm-up and 8 tail rows of a segment are being read by its neighbour at that
    // moment (L2 hits instead of a second trip to DRAM).  The kernel is symmetric in the row direction (symmetric taps, symmetric
    // Laplacian): `lrow(k)` maps the logical row k of the walk to the image row.  The tap sums of an up-walking segment run in the
    // opposite row order (last-ulp differences), which is why seg_rows is a constant of the launch geometry: the direction of a
    // row depends on the frame height only, never on the batch.
    const int dir = (seg & 1) ? -1 : 1;
    const int base = (seg & 1) ? r1 - 1 : r0;
    auto lrow = [&](int k) { return base + dir * k; };
    const int c0 = band * kSsBandCols - kSsLaneCols + lane * kSsLaneCols;   // plane column of this lane's first pixel
    const long long plane = (long long)h * w;
    const float* img = x + (long long)f * 3 * plane + min(max(c0, 0), w - kSsLaneCols);
    const bool writer = lane >= 1 && lane <= 30 && c0 < w;
    const bool left_edge = band == 0;                       // lane 0 holds columns -8 .. -1
    const int lane_r = (w - band * kSsBandCols) / kSsLaneCols + 1;   // the lane that holds columns w .. w+7 (if <= 31)
    const bool right_edge = lane_r <= 31;

    const uint32_t ring0 = uint32_t(__cvta_generic_to_shared(s_ring)) + uint32_t(lane) * 16u;
    f32x2 T[8];
#pragma unroll
    for (int d = 0; d < 8; ++d) T[d] = pk2(taps.t[d], taps.t[d]);

    f32x2 gm2[4], gm1[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) gm2[j] = gm1[j] = 0ull;
    float mn = INFINITY, mx = -INFINITY;

    auto row_ptr = [&](int k) -> const float* {
        k = k < 0 ? -k : (k >= h ? 2 * (h - 1) - k : k);      // BORDER_REFLECT_101, |overhang| <= 10 < h
        return img + (long long)k * w;
    };
    float4 nx[2][3][2];
    auto load_rows = [&](int k) {      // logical rows k, k + 1
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const float* rp = row_ptr(lrow(k + rr));
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                nx[rr][c][0] = __ldg(reinterpret_cast<const float4*>(rp + c * plane));
                nx[rr][c][1] = __ldg(reinterpret_cast<const float4*>(rp + c * plane) + 1);
            }
        }
    };
    auto prefetch_rows = [&](int k) {
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const float* rp = row_ptr(lrow(k + rr));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(rp));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + plane));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + 2 * plane));
        }
    };
    // gray of one loaded row (packed column pairs) incl. the reflected halo columns at the image borders
    auto gray_row = [&](const float4 (&v)[3][2], f32x2 (&out)[4], int k) {
        const float r[8] = {v[0][0].x, v[0][0].y, v[0][0].z, v[0][0].w, v[0][1].x, v[0][1].y, v[0][1].z, v[0][1].w};
        const float g[8] = {v[1][0].x, v[1][0].y, v[1][0].z, v[1][0].w, v[1][1].x, v[1][1].y, v[1][1].z, v[1][1].w};
        const float b[8] = {v[2][0].x, v[2][0].y, v[2][0].z, v[2][0].w, v[2][1].x, v[2][1].y, v[2][1].z, v[2][1].w};
        if constexpr (kLum) {
            if (writer && k >= r0 && k < r1) {      // rows of this segment only (never a reflected row)
                float l[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) l[i] = __fadd_rn(__fadd_rn(__fmul_rn(0.299f, r[i]), __fmul_rn(0.587f, g[i])), __fmul_rn(0.114f, b[i]));
                float* dst = lum_out + (long long)f * lum_stride + (long long)k * w + c0;
                __stcg(reinterpret_cast<float4*>(dst), make_float4(l[0], l[1], l[2], l[3]));
                __stcg(reinterpret_cast<float4*>(dst + 4), make_float4(l[4], l[5], l[6], l[7]));
            }
        }
        s2_gray8(r, g, b, out);
        if (left_edge || right_edge) {      // warp-uniform
            float e[8], o[8];
#pragma unroll
            for (int j = 0; j < 4; ++j) upk2(out[j], e[2 * j], e[2 * j + 1]);
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = e[i];
            if (left_edge) {
                // column -8 + i  <-  column 8 - i : lane 2 element 0 (i = 0), lane 1 element 8 - i (i = 1 .. 7)
                const float t0 = __shfl_sync(0xffffffffu, e[0], 2);
                if (lane == 0) o[0] = t0;
#pragma unroll
                for (int i = 1; i < 8; ++i) {
                    const float ti = __shfl_sync(0xffffffffu, e[8 - i], 1);
                    if (lane == 0) o[i] = ti;
                }
            }
            if (right_edge) {
                // column w + j  <-  column w - 2 - j : lane_r - 1 element 6 - j (j = 0 .. 6), lane_r - 2 element 7 (j = 7)
#pragma unroll
                for (int j = 0; j < 7; ++j) {
                    const float tj = __shfl_sync(0xffffffffu, e[6 - j], (lane_r - 1) & 31);
                    if (lane == lane_r) o[j] = tj;
                }
                const float t7 = __shfl_sync(0xffffffffu, e[7], (lane_r - 2) & 31);
                if (lane == lane_r) o[7] = t7;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) out[j] = pk2(o[2 * j], o[2 * j + 1]);
        }
    };

    // (logical rows of the walk) iteration t converts gray rows G0 + 2t, G0 + 2t + 1, forms |lap| rows G0 + 2t - 1, G0 + 2t and,
    // from t = 8 on, the output rows m = 2 (t - 8) and m + 1 (|lap| rows m - 7 .. m + 8 are then in the ring)
    const int G0 = -8;
    const int iters = 8 + (r1 - r0 + 1) / 2;
    load_rows(G0);
    uint32_t p = 0;   // ring row that receives the first of this iteration's two |lap| rows (even)
#pragma unroll 1
    for (int t = 0; t < iters; ++t) {
        f32x2 ga[4], gb[4];
        gray_row(nx[0], ga, lrow(G0 + 2 * t));
        gray_row(nx[1], gb, lrow(G0 + 2 * t + 1));
        if (t + 1 < iters) load_rows(G0 + 2 * (t + 1));
        if (t + 2 < iters) prefetch_rows(G0 + 2 * (t + 2));
        float la[8], lb[8];
        s2_lap8(gm2, gm1, ga, la);
        s2_lap8(gm1, ga, gb, lb);
        uint32_t ha[4], hb[4];       // the two new |lap| rows as fp16 pairs
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const __half2 a2 = __floats2half2_rn(la[2 * j], la[2 * j + 1]), b2 = __floats2half2_rn(lb[2 * j], lb[2 * j + 1]);
            ha[j] = *reinterpret_cast<const uint32_t*>(&a2);
            hb[j] = *reinterpret_cast<const uint32_t*>(&b2);
        }
        {
            const uint32_t a0 = ring0 + p * uint32_t(kS2RingRowBytes);
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(a0), "r"(ha[0]), "r"(ha[1]), "r"(ha[2]), "r"(ha[3]) : "memory");
            asm volatile("st.shared.v4.b32 [%0+512], {%1,%2,%3,%4};" ::"r"(a0), "r"(hb[0]), "r"(hb[1]), "r"(hb[2]), "r"(hb[3]) : "memory");
        }
        if (t >= 8) {
            // ---- vertical pass of rows m (taps |i - 7|) and m + 1 (taps |i - 8|) over |lap| rows m - 7 + i, i = 0 .. 15: rows
            // 0 .. 13 stream from the fp16 ring (one 128-bit load per row and lane), rows 14 and 15 are this iteration's own
            // registers.  (Keeping 4 .. 12 more rows in registers across iterations changes nothing: 0.61-0.63 ms either way --
            // with the luma plane written as well the kernel moves 3.0 GB per 16 x 4K in 0.48 ms, i.e. it runs at the HBM rate) ----
            f32x2 am[4], am1[4];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                f32x2 v[4];
                if (i < 14) {
                    uint32_t u[4];
                    const uint32_t a = ring0 + (((p + 2u + uint32_t(i)) & 15u) * uint32_t(kS2RingRowBytes));
                    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]) : "r"(a));
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&u[j]));
                        v[j] = pk2(c.x, c.y);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[j] = i == 14 ? pk2(la[2 * j], la[2 * j + 1]) : pk2(lb[2 * j], lb[2 * j + 1]);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (i == 0) am[j] = mul2(T[7], v[j]);
                    else if (i <= 14) am[j] = fma2(T[i < 7 ? 7 - i : i - 7], v[j], am[j]);
                    if (i == 1) am1[j] = mul2(T[7], v[j]);
                    else if (i >= 2) am1[j] = fma2(T[i < 8 ? 8 - i : i - 8], v[j], am1[j]);
                }
            }
            // ---- exchange the two rows of vertical sums with the neighbouring lanes ----
            float* xr0 = s_xch[t & 1][0];
            float* xr1 = s_xch[t & 1][1];
            {
                const uint32_t b0 = uint32_t(__cvta_generic_to_shared(xr0)) + uint32_t(lane + 1) * 16u;
                const uint32_t b1 = uint32_t(__cvta_generic_to_shared(xr1)) + uint32_t(lane + 1) * 16u;
                asm volatile("st.shared.v2.b64 [%0], {%1,%2};" ::"r"(b0), "l"(am[0]), "l"(am[1]) : "memory");
                asm volatile("st.shared.v2.b64 [%0+544], {%1,%2};" ::"r"(b0), "l"(am[2]), "l"(am[3]) : "memory");
                asm volatile("st.shared.v2.b64 [%0], {%1,%2};" ::"r"(b1), "l"(am1[0]), "l"(am1[1]) : "memory");
                asm volatile("st.shared.v2.b64 [%0+544], {%1,%2};" ::"r"(b1), "l"(am1[2]), "l"(am1[3]) : "memory");
            }
            __syncwarp();
            const int m = 2 * (t - 8);
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
                const float4* rowA = reinterpret_cast<const float4*>(rr == 0 ? xr0 : xr1) + 1;   // slot -1 and slot 32 are padding
                const float4* rowB = rowA + 34;
                float bwin[24];
                {
                    const float4 t0 = rowA[lane - 1], t1 = rowB[lane - 1], t4 = rowA[lane + 1], t5 = rowB[lane + 1];
                    bwin[0] = t0.x; bwin[1] = t0.y; bwin[2] = t0.z; bwin[3] = t0.w;
                    bwin[4] = t1.x; bwin[5] = t1.y; bwin[6] = t1.z; bwin[7] = t1.w;
#pragma unroll
                    for (int j = 0; j < 4; ++j) upk2(rr == 0 ? am[j] : am1[j], bwin[8 + 2 * j], bwin[9 + 2 * j]);
                    bwin[16] = t4.x; bwin[17] = t4.y; bwin[18] = t4.z; bwin[19] = t4.w;
                    bwin[20] = t5.x; bwin[21] = t5.y; bwin[22] = t5.z; bwin[23] = t5.w;
                }
                // horizontal pass: symmetric pair sums are scalar adds into aligned register pairs, the tap FMAs are packed
                float o[8];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int i = 2 * j;
                    f32x2 acc = mul2(T[0], pk2(bwin[8 + i], bwin[9 + i]));
#pragma unroll
                    for (int d = 1; d <= 7; ++d)
                        acc = fma2(T[d], pk2(__fadd_rn(bwin[8 + i - d], bwin[8 + i + d]), __fadd_rn(bwin[9 + i - d], bwin[9 + i + d])), acc);
                    upk2(acc, o[i], o[i + 1]);
                }
                const int row = lrow(m + rr);
                if (writer && m + rr < r1 - r0) {
                    float* dst = blur_out + (long long)f * plane + (long long)row * w + c0;
                    __stcg(reinterpret_cast<float4*>(dst), make_float4(o[0], o[1], o[2], o[3]));
                    __stcg(reinterpret_cast<float4*>(dst + 4), make_float4(o[4], o[5], o[6], o[7]));
#pragma unroll
                    for (int i = 0; i < 8; i += 2) { mn = fminf(mn, fminf(o[i], o[i + 1])); mx = fmaxf(mx, fmaxf(o[i], o[i + 1])); }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) { gm2[j] = ga[j]; gm1[j] = gb[j]; }
        p = (p + 2u) & 15u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0 && mn <= mx) {
        atomicMin(&mm[f].blur_min, dbl_key(double(mn)));
        atomicMax(&mm[f].blur_max, dbl_key(double(mx)));
    }
}

// sal = float((blur - min) / (max - min + 1e-8)); optional attention raw value + its fp32 min/max.
// blur is held in fp32 (so min and max are fp32 values).  Per pixel: one fp32 subtraction, one multiplication by the per-image
// reciprocal of the range (formed once per thread in fp64) and, for the attention, one multiplication by rcp.approx(luma + 0.1):
// within ~3 ulp of the reference's quotients -- 4e-7 on maps normalised to [0,1], against a stated bound of 1e-4 (SURVEY 8c; the
// full-map oracle tests hold 2e-6) -- instead of two IEEE divisions and an fp64 round trip per pixel, which kept this kernel on
// the XU pipe (ncu round 3: 43-46 %) instead of on its memory streams.  VEC = 4 pixels per thread.
__device__ __forceinline__ float rcp_approx(float v)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}

// kLumPlane: `x` is a luma plane left behind by k_saliency_stream2<true> (frame stride x_stride floats) instead of the RGB frame.
template <bool kAttention, int VEC, bool kLumPlane = false>
__global__ void __launch_bounds__(kSalThreads)
k_sal_normalize(const float* __restrict__ blur, const float* __restrict__ x, float* __restrict__ out, long long plane,
                SalMinMax* __restrict__ mm, long long x_stride = 0)
{
    __shared__ float s_mn[kSalThreads / 32], s_mx[kSalThreads / 32];
    const int f = blockIdx.y;
    const double bmn = key_dbl(mm[f].blur_min), bmx = key_dbl(mm[f].blur_max);
    const float bmn_f = float(bmn);                       // exact: the minimum of fp32 values
    const float inv_den = float(1.0 / (bmx - bmn + 1e-8));
    const float* img = x + (long long)f * (kLumPlane ? x_stride : 3 * plane);
    const float* bl = blur + (long long)f * plane;
    float* o = out + (long long)f * plane;
    float mn = INFINITY, mx = -INFINITY;
    const long long nvec = plane / VEC;
    const long long stride = (long long)gridDim.x * kSalThreads;
    for (long long i = (long long)blockIdx.x * kSalThreads + threadIdx.x; i < nvec; i += stride) {
        float b[VEC], r[VEC], g[VEC], bb[VEC], res[VEC];
        if (VEC == 4) {
            const float4 t = __ldcs(reinterpret_cast<const float4*>(bl) + i);
            b[0] = t.x; b[1] = t.y; b[2] = t.z; b[3] = t.w;
            if (kAttention && kLumPlane) {
                const float4 tl = __ldcs(reinterpret_cast<const float4*>(img) + i);
                r[0] = tl.x; r[1] = tl.y; r[2] = tl.z; r[3] = tl.w;
            } else if (kAttention) {
                const float4 tr = __ldg(reinterpret_cast<const float4*>(img) + i);
                const float4 tg = __ldg(reinterpret_cast<const float4*>(img + plane) + i);
                const float4 tb = __ldg(reinterpret_cast<const float4*>(img + 2 * plane) + i);
                r[0] = tr.x; r[1] = tr.y; r[2] = tr.z; r[3] = tr.w;
                g[0] = tg.x; g[1] = tg.y; g[2] = tg.z; g[3] = tg.w;
                bb[0] = tb.x; bb[1] = tb.y; bb[2] = tb.z; bb[3] = tb.w;
            }
        } else {
            b[0] = bl[i];
            if (kAttention) { r[0] = __ldg(img + i); g[0] = __ldg(img + plane + i); bb[0] = __ldg(img + 2 * plane + i); }
        }
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            const float sal = __fmul_rn(__fsub_rn(b[k], bmn_f), inv_den);
            if (kAttention) {
                const float lum = kLumPlane ? r[k]
                                            : __fadd_rn(__fadd_rn(__fmul_rn(0.299f, r[k]), __fmul_rn(0.587f, g[k])), __fmul_rn(0.114f, bb[k]));
                const float a = __fmul_rn(sal, rcp_approx(__fadd_rn(lum, 0.1f)));
                res[k] = a;
                mn = fminf(mn, a);
                mx = fmaxf(mx, a);
            } else {
                res[k] = sal;
            }
        }
        if (VEC == 4) reinterpret_cast<float4*>(o)[i] = make_float4(res[0], res[1], res[2], res[3]);
        else o[i] = res[0];
    }
    if constexpr (kAttention) {
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, sh));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, sh));
    }
    if ((threadIdx.x & 31) == 0) { s_mn[threadIdx.x >> 5] = mn; s_mx[threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 1; k < kSalThreads / 32; ++k) { mn = fminf(mn, s_mn[k]); mx = fmaxf(mx, s_mx[k]); }
        if (mn <= mx) {
            atomicMin(&mm[f].att_min, flt_key(mn));
            atomicMax(&mm[f].att_max, flt_key(mx));
        }
    }
    }
}

// 1 / (max - min + 1e-8) of the raw attention (content_aware.py:88-89), once per thread: the per-pixel quotient becomes a product
__device__ __forceinline__ float att_inv_range(float mn, float mx)
{
    return __fdiv_rn(1.0f, __fadd_rn(__fsub_rn(mx, mn), 1e-8f));
}

template <int VEC>
__global__ void __launch_bounds__(kSalThreads)
k_att_normalize(float* __restrict__ att, long long plane, const SalMinMax* __restrict__ mm)
{
    const int f = blockIdx.y;
    const float mn = key_flt(mm[f].att_min), mx = key_flt(mm[f].att_max);
    const float inv = att_inv_range(mn, mx);
    const long long nvec = plane / VEC;
    const long long stride = (long long)gridDim.x * kSalThreads;
    float* base = att + (long long)f * plane;
    for (long long i = (long long)blockIdx.x * kSalThreads + threadIdx.x; i < nvec; i += stride) {
        if (VEC == 4) {
            float4 v = reinterpret_cast<float4*>(base)[i];
            v.x = __fmul_rn(__fsub_rn(v.x, mn), inv);
            v.y = __fmul_rn(__fsub_rn(v.y, mn), inv);
            v.z = __fmul_rn(__fsub_rn(v.z, mn), inv);
            v.w = __fmul_rn(__fsub_rn(v.w, mn), inv);
            reinterpret_cast<float4*>(base)[i] = v;
        } else {
            base[i] = __fmul_rn(__fsub_rn(base[i], mn), inv);
        }
    }
}

// a7 in one pass over the raw attention: att = (raw - min) / (max - min + 1e-8); out = clamp(enh * (1 + 0.2 att), 0, 1)
// (content_aware.py:88-90 and :119-120).  One item = 4 pixels of one frame, all three channels: the raw attention is read
// once instead of being normalised in place (8 B/px) and then re-read per channel by the gain kernel.
__device__ __forceinline__ float sal_clamp01_keep_nan(float v) { return v < 0.0f ? 0.0f : (v > 1.0f ? 1.0f : v); }

// kGain: the multi-scale gain of the same input (multi_scale.py:97-98) is applied in the same epilogue, to the clamped
// content-aware result: out = clamp(clamp(enh * (1 + 0.2 att), 0, 1) * gain[f], 0, 1) -- the "content-aware + multi-scale"
// chain of BASELINE config 5 without a second pass over the frame.
template <bool kWriteAtt, bool kGain, int VEC>
__global__ void __launch_bounds__(kSalThreads)
k_att_gain(const float* __restrict__ raw, const float* __restrict__ enh, float* __restrict__ out, float* __restrict__ att_out,
           long long plane, const SalMinMax* __restrict__ mm, const float* __restrict__ gain)
{
    const int f = blockIdx.y;
    const float ms_gain = kGain ? __ldg(gain + f) : 1.0f;
    const float mn = key_flt(mm[f].att_min), mx = key_flt(mm[f].att_max);
    const float inv = att_inv_range(mn, mx);
    const float* r = raw + (long long)f * plane;
    const float* e = enh + (long long)f * 3 * plane;
    float* o = out + (long long)f * 3 * plane;
    float* ao = kWriteAtt ? att_out + (long long)f * plane : nullptr;
    const long long nvec = plane / VEC;
    const long long stride = (long long)gridDim.x * kSalThreads;
#pragma unroll 2
    for (long long i = (long long)blockIdx.x * kSalThreads + threadIdx.x; i < nvec; i += stride) {
        float a[VEC], g[VEC];
        if (VEC == 4) {
            const float4 t = __ldcs(reinterpret_cast<const float4*>(r) + i);
            a[0] = t.x; a[1] = t.y; a[2] = t.z; a[3] = t.w;
        } else {
            a[0] = r[i];
        }
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            a[k] = __fmul_rn(__fsub_rn(a[k], mn), inv);
            g[k] = __fadd_rn(1.0f, __fmul_rn(0.2f, a[k]));
        }
        if (kWriteAtt) {
            if (VEC == 4) reinterpret_cast<float4*>(ao)[i] = make_float4(a[0], a[1], a[2], a[3]);
            else ao[i] = a[0];
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            if (VEC == 4) {
                const float4 v = __ldcs(reinterpret_cast<const float4*>(e + c * plane) + i);
                float4 w;
                w.x = sal_clamp01_keep_nan(__fmul_rn(v.x, g[0]));
                w.y = sal_clamp01_keep_nan(__fmul_rn(v.y, g[1]));
                w.z = sal_clamp01_keep_nan(__fmul_rn(v.z, g[2]));
                w.w = sal_clamp01_keep_nan(__fmul_rn(v.w, g[3]));
                if (kGain) {
                    w.x = sal_clamp01_keep_nan(__fmul_rn(w.x, ms_gain));
                    w.y = sal_clamp01_keep_nan(__fmul_rn(w.y, ms_gain));
                    w.z = sal_clamp01_keep_nan(__fmul_rn(w.z, ms_gain));
                    w.w = sal_clamp01_keep_nan(__fmul_rn(w.w, ms_gain));
                }
                __stcs(reinterpret_cast<float4*>(o + c * plane) + i, w);
            } else {
                float w1 = sal_clamp01_keep_nan(__fmul_rn(e[c * plane + i], g[0]));
                if (kGain) w1 = sal_clamp01_keep_nan(__fmul_rn(w1, ms_gain));
                o[c * plane + i] = w1;
            }
        }
    }
}

// The attention gain of the map epilogue: the k_att_gain<false, false> arithmetic over the raw attention plane and its min/max
struct AttGain {
    const float* raw;
    const SalMinMax* mm;
    long long plane;
    static constexpr bool kApply = true;
    struct Frame {
        const float* r;
        float mn, inv;
        __device__ float gain(float a) const { return __fadd_rn(1.0f, __fmul_rn(0.2f, __fmul_rn(__fsub_rn(a, mn), inv))); }
        __device__ float4 g4(long long q) const
        {
            const float4 t = __ldcs(reinterpret_cast<const float4*>(r) + q);
            return make_float4(gain(t.x), gain(t.y), gain(t.z), gain(t.w));
        }
        __device__ float g1(long long p) const { return gain(r[p]); }
    };
    __device__ Frame frame(int f) const
    {
        const float mn = key_flt(mm[f].att_min), mx = key_flt(mm[f].att_max);
        return {raw + f * plane, mn, att_inv_range(mn, mx)};
    }
};

static GaussTapsF sal_taps_f()
{
    // cv2.getGaussianKernel(15, sigma=0.3*((15-1)*0.5-1)+0.8 = 2.6) in fp64, rounded to fp32; t[d] = weight at distance d
    double k[15], sum = 0.0;
    const double sigma = 0.3 * ((15 - 1) * 0.5 - 1) + 0.8;
    for (int i = 0; i < 15; ++i) { const double d = i - 7; k[i] = std::exp(-0.5 * d * d / (sigma * sigma)); sum += k[i]; }
    GaussTapsF r;
    for (int d = 0; d < 8; ++d) r.t[d] = float(k[7 + d] / sum);
    return r;
}

static size_t sal_ws_bytes(int n, int h, int w)
{
    return align_up(size_t(n) * sizeof(SalMinMax), 256) + align_up(size_t(n) * h * w * sizeof(float), 256);
}

// mode 0: saliency only -> out ; mode 1: attention -> out (saliency is an internal temporary);
// mode 2: out = clamp(enh * (1 + 0.2 attention), 0, 1) with the attention map optional (att_out)
// The passes of one (sub-)batch of n frames on stream s.  mm / blur: the min-max records and the intermediate plane of these frames.
// lum_ok: the result frame may serve as luma scratch (mode 2, no aliasing with the inputs).
// maps (mode 2): the result is the map epilogue of these frames (out is maps->out, enh is unused).
static int sal_launch(int mode, const float* x, int n, int h, int w, float* out, SalMinMax* mm, float* blur, cudaStream_t s,
                      const float* enh, float* att_out, const float* ms_gain, bool lum_ok, const MapsArgs* maps)
{
    const long long plane = (long long)h * w;
    k_sal_reset<<<(n + 127) / 128, 128, 0, s>>>(mm, n);
    UPR_LAUNCH_CHECK();
    bool lum_in_out = false;
    {
        static const GaussTapsF taps = sal_taps_f();
        const int bands = (w + kSsBandCols - 1) / kSsBandCols;
        // one warp per (band, row segment, frame).  General kernel: aim at ~6 warps per resident slot (20 warps/SM) for balance, but
        // keep segments >= 64 rows (16 of every segment's rows are re-computed halo; segments of 96 / 128 / 192 rows leave too few
        // warps: content-aware op 1.31 -> 1.34 / 1.38 / 1.43 ms per 16 x 4K)
        const long long slots = 18LL * kNumSMsB200;
        long long nseg = (6 * slots + (long long)n * bands - 1) / ((long long)n * bands);
        nseg = std::max<long long>(1, std::min<long long>(nseg, (h + 63) / 64));
        // the packed two-rows-per-iteration kernel serves w % 8 == 0, h >= 16, 16-byte aligned planes; everything else (ragged
        // widths, tiny images, unaligned views) takes the general one-row kernel with its reflect-indexed scalar loads
        // (w >= 16, h >= 16: one reflection must bring every halo column / row back inside the image)
        const bool packed = w % 8 == 0 && w >= 16 && h >= 16 && aligned16(x) && aligned16(blur);
        // packed kernel: 64-row segments whatever the batch (its odd segments walk upwards: a row's direction, hence the last ulp of
        // its tap sums, must not depend on n)
        const int seg_rows = packed ? kS2SegRows : int((h + nseg - 1) / nseg);
        const int segs = (h + seg_rows - 1) / seg_rows;
        if ((long long)bands * segs > 0x7fffffffLL) return UPR_E_SHAPE;
        // content-aware apply: the result frame is free scratch until the last pass writes it -- its first plane takes luma(x),
        // which the attention pass then reads instead of the 12 B/px frame (not when `out` aliases an input)
        lum_in_out = packed && mode == 2 && lum_ok && aligned16(out);
        if (packed && lum_in_out)
            k_saliency_stream2<true><<<dim3(unsigned(bands * segs), n), 32, 0, s>>>(x, h, w, bands, seg_rows, blur, mm, taps, out, 3 * plane);
        else if (packed)
            k_saliency_stream2<false><<<dim3(unsigned(bands * segs), n), 32, 0, s>>>(x, h, w, bands, seg_rows, blur, mm, taps, nullptr, 0);
        else k_saliency_stream<<<dim3(unsigned(bands * segs), n), 32, 0, s>>>(x, h, w, bands, seg_rows, blur, mm, taps);
    }
    UPR_LAUNCH_CHECK();
    const bool v4 = plane % 4 == 0 && aligned16(x) && aligned16(out) && (mode != 2 || (aligned16(enh) && (!att_out || aligned16(att_out))));
    const long long work = v4 ? plane / 4 : plane;
    const int parts = int(std::max<long long>(1, std::min<long long>((work + kSalThreads * 2 - 1) / (kSalThreads * 2),
                                                                     (16LL * kNumSMsB200 + n - 1) / n)));
    if (mode == 0) {
        if (v4) k_sal_normalize<false, 4><<<dim3(parts, n), kSalThreads, 0, s>>>(blur, x, out, plane, mm);
        else k_sal_normalize<false, 1><<<dim3(parts, n), kSalThreads, 0, s>>>(blur, x, out, plane, mm);
        UPR_LAUNCH_CHECK();
    } else if (mode == 2) {
        // raw attention over the blur plane in place (each element is read and written by the same thread)
        if (lum_in_out) k_sal_normalize<true, 4, true><<<dim3(parts, n), kSalThreads, 0, s>>>(blur, out, blur, plane, mm, 3 * plane);
        else if (v4) k_sal_normalize<true, 4><<<dim3(parts, n), kSalThreads, 0, s>>>(blur, x, blur, plane, mm);
        else k_sal_normalize<true, 1><<<dim3(parts, n), kSalThreads, 0, s>>>(blur, x, blur, plane, mm);
        UPR_LAUNCH_CHECK();
        if (maps) return maps_epilogue(*maps, n, h, w, AttGain{blur, mm, plane}, s);
        const dim3 grid(parts, n);
#define UPR_ATT_GAIN(A, G)                                                                                                     \
    do {                                                                                                                       \
        if (v4) k_att_gain<A, G, 4><<<grid, kSalThreads, 0, s>>>(blur, enh, out, att_out, plane, mm, ms_gain);                  \
        else k_att_gain<A, G, 1><<<grid, kSalThreads, 0, s>>>(blur, enh, out, att_out, plane, mm, ms_gain);                     \
    } while (0)
        if (att_out && ms_gain) UPR_ATT_GAIN(true, true);
        else if (att_out) UPR_ATT_GAIN(true, false);
        else if (ms_gain) UPR_ATT_GAIN(false, true);
        else UPR_ATT_GAIN(false, false);
#undef UPR_ATT_GAIN
        UPR_LAUNCH_CHECK();
    } else {
        if (v4) k_sal_normalize<true, 4><<<dim3(parts, n), kSalThreads, 0, s>>>(blur, x, out, plane, mm);
        else k_sal_normalize<true, 1><<<dim3(parts, n), kSalThreads, 0, s>>>(blur, x, out, plane, mm);
        UPR_LAUNCH_CHECK();
        if (v4) k_att_normalize<4><<<dim3(parts, n), kSalThreads, 0, s>>>(out, plane, mm);
        else k_att_normalize<1><<<dim3(parts, n), kSalThreads, 0, s>>>(out, plane, mm);
        UPR_LAUNCH_CHECK();
    }
    return UPR_OK;
}


// Multi-scale statistics of the same frames, computed inside the schedule (BASELINE config 5 chain): the statistics kernel of a
// chunk runs on the chunk's stream ahead of its blur kernel, so its issue-bound pass overlaps the memory-bound passes of the
// neighbouring chunk instead of running alone over the whole batch first.
struct MsJob {
    MsStreamGeom geo;
    void* ws;
    size_t ws_bytes;
    float* means3;      // [n][3]
    float* gain;        // [n]
};

// maps (mode 2): the content-aware result of the CNN maps -- pass 3 is the map epilogue with the attention gain; out must be
// maps->out (NULL for the u8 result) and enh NULL.
static int sal_run(int mode, const float* x, int n, int h, int w, float* out, void* ws, size_t ws_bytes, cudaStream_t s,
                   const float* enh = nullptr, float* att_out = nullptr, const float* ms_gain = nullptr, const MsJob* ms = nullptr,
                   const MapsArgs* maps = nullptr)
{
    if (n < 0 || n > 65535 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    if (n == 0) return UPR_OK;
    if (!x || !(out || maps) || !ws || (mode == 2 && !enh && !maps)) return UPR_E_NULL;
    if (ws_bytes < sal_ws_bytes(n, h, w) || (reinterpret_cast<uintptr_t>(ws) & 255u)) return UPR_E_WORKSPACE;
    auto* mm = static_cast<SalMinMax*>(ws);
    auto* blur = reinterpret_cast<float*>(static_cast<unsigned char*>(ws) + align_up(size_t(n) * sizeof(SalMinMax), 256));
    const long long plane = (long long)h * w;
    // lum_ok: the f32 result frame is luma scratch between the passes, which it may be unless it aliases an input (in-place
    // apply).  chunk_ok: the frames may run chunk by chunk on the side streams.  A u8 result cannot hold luma (3 < 4 B/px) and
    // aliases no f32 input, so it chunks without the scratch.
    bool lum_ok = false, chunk_ok = true;
    if (mode == 2 && out) {
        const size_t frame_bytes = size_t(n) * 3 * plane * sizeof(float);
        const char *o0 = reinterpret_cast<const char*>(out), *o1 = o0 + frame_bytes;
        auto overlaps = [&](const void* q, size_t bytes) {
            const char* q0 = reinterpret_cast<const char*>(q);
            return q0 < o1 && q0 + bytes > o0;
        };
        lum_ok = !overlaps(x, frame_bytes) &&
                 (maps ? !overlaps(maps->illu, size_t(n) * plane * map_dtype_bytes(maps->illu_dt)) &&
                             !overlaps(maps->e, frame_bytes / sizeof(float) * map_dtype_bytes(maps->e_dt))
                       : !overlaps(enh, frame_bytes));
        chunk_ok = lum_ok;
    }
    // Chunked schedule: the three passes of a chunk of ~25 Mpx run back to back on one of two side streams, consecutive chunks on
    // alternating streams.  The 4-8 B/px intermediate of a chunk (~100-200 MB) is then re-read while part of it is still in L2, and
    // the passes of neighbouring chunks overlap.  Measured on 16 x 4K / 64 x 1080p: 1.39 -> 1.28-1.30 ms (profiles/r4_content_aware.md;
    // single-frame chunks lose more to short kernels than they gain).  Results do not depend on the schedule: every frame is
    // normalised on its own.  An in-place apply (!chunk_ok) runs as one chunk.
    const int chunk = chunk_ok ? chunk_frames(plane) : n;
    const long long step_x = 3 * plane, step_p = plane;
    return run_chunked(s, n, chunk, [&](int f0, int nf, cudaStream_t cs) {
        if (ms) {
            const int rc = ms_stream_launch_range(x + f0 * step_x, nf, h, w, ms->geo, ms->ws, ms->ws_bytes, n, f0, ms->means3 + 3 * f0,
                                                  ms->gain + f0, cs);
            if (rc != UPR_OK) return rc;
        }
        const MapsArgs mf = maps ? maps->at(f0, plane) : MapsArgs{};
        return sal_launch(mode, x + f0 * step_x, nf, h, w, out ? out + f0 * (mode == 2 ? step_x : step_p) : nullptr, mm + f0,
                          blur + f0 * step_p, cs, enh ? enh + f0 * step_x : nullptr, att_out ? att_out + f0 * step_p : nullptr,
                          ms_gain ? ms_gain + f0 : nullptr, lum_ok, maps ? &mf : nullptr);
    });
}

}  // namespace upr

extern "C" {

size_t upr_saliency_workspace_bytes(int n, int h, int w)
{
    if (n < 0 || h <= 0 || w <= 0) return 0;
    return upr::sal_ws_bytes(std::max(n, 1), h, w);
}

int upr_saliency_f32(const float* x_nchw, int n, int h, int w, float* sal_n1hw, void* workspace, size_t workspace_bytes,
                     upr_stream_t stream)
{
    return upr::sal_run(0, x_nchw, n, h, w, sal_n1hw, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int upr_attention_f32(const float* x_nchw, int n, int h, int w, float* att_n1hw, void* workspace, size_t workspace_bytes,
                      upr_stream_t stream)
{
    return upr::sal_run(1, x_nchw, n, h, w, att_n1hw, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int upr_content_aware_apply_f32(const float* x_nchw, const float* enh_nchw, float* out_nchw, float* att_n1hw, int n, int h,
                                int w, void* workspace, size_t workspace_bytes, upr_stream_t stream)
{
    return upr::sal_run(2, x_nchw, n, h, w, out_nchw, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), enh_nchw,
                        att_n1hw);
}

int upr_content_multiscale_f32(const float* x_nchw, const float* enh_nchw, float* out_nchw, float* att_n1hw, float* means_n_by_3,
                               float* gain_per_image, int n, int h, int w, void* workspace, size_t workspace_bytes,
                               void* ms_workspace, size_t ms_workspace_bytes, upr_stream_t stream)
{
    if (n > 0 && (!means_n_by_3 || !gain_per_image || !ms_workspace)) return UPR_E_NULL;
    auto s = static_cast<cudaStream_t>(stream);
    upr::MsStreamGeom geo{};
    // shapes the streaming statistics kernel does not serve: the generic statistics path over the whole batch first
    if (n > 0 && !upr::ms_stream_geometry(h, w, x_nchw, &geo)) {
        const int rc = upr_multiscale_stats_f32(x_nchw, n, h, w, means_n_by_3, gain_per_image, ms_workspace, ms_workspace_bytes, 0, stream);
        if (rc) return rc;
        return upr::sal_run(2, x_nchw, n, h, w, out_nchw, workspace, workspace_bytes, s, enh_nchw, att_n1hw, gain_per_image);
    }
    const upr::MsJob job{geo, ms_workspace, ms_workspace_bytes, means_n_by_3, gain_per_image};
    return upr::sal_run(2, x_nchw, n, h, w, out_nchw, workspace, workspace_bytes, s, enh_nchw, att_n1hw, gain_per_image, &job);
}

int upr_retinex_content_aware_typed_f32(const float* x_nchw, const void* illu_n1hw, int illu_dtype, const void* e_nchw, int e_dtype,
                                        int flags, float* out_nchw, int n, int h, int w, float eps, void* workspace,
                                        size_t workspace_bytes, upr_stream_t stream)
{
    if (n < 0 || n > 65535 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    const upr::MapsArgs m{x_nchw, illu_n1hw, illu_dtype, e_nchw, e_dtype, flags, eps, out_nchw, nullptr, nullptr};
    bool done;
    const int rc = upr::maps_check(m, n, &done);
    if (done) return rc;
    return upr::sal_run(2, x_nchw, n, h, w, out_nchw, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), nullptr, nullptr,
                        nullptr, nullptr, &m);
}

int upr_retinex_content_aware_typed_u8(const float* x_nchw, const void* illu_n1hw, int illu_dtype, const void* e_nchw, int e_dtype,
                                       int flags, unsigned char* out_nhwc, unsigned char* illu_nhw1, int n, int h, int w, float eps,
                                       void* workspace, size_t workspace_bytes, upr_stream_t stream)
{
    if (n < 0 || n > 65535 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    const upr::MapsArgs m{x_nchw, illu_n1hw, illu_dtype, e_nchw, e_dtype, flags, eps, nullptr, out_nhwc, illu_nhw1};
    bool done;
    const int rc = upr::maps_check(m, n, &done);
    if (done) return rc;
    return upr::sal_run(2, x_nchw, n, h, w, nullptr, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), nullptr, nullptr,
                        nullptr, nullptr, &m);
}

int upr_content_multiscale_apply_f32(const float* x_nchw, const float* enh_nchw, const float* ms_gain_per_image, float* out_nchw,
                                     float* att_n1hw, int n, int h, int w, void* workspace, size_t workspace_bytes,
                                     upr_stream_t stream)
{
    if (!ms_gain_per_image && n > 0) return UPR_E_NULL;
    return upr::sal_run(2, x_nchw, n, h, w, out_nchw, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), enh_nchw,
                        att_n1hw, ms_gain_per_image);
}

}  // extern "C"
