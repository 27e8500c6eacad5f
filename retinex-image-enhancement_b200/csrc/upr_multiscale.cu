// upr_multiscale.cu -- three-scale feature statistics and gain of the multi-scale enhancer (sm_100a).
//
// Replaces MultiScaleEnhancer.extract_multi_scale_features and the gain computation of
// apply_multi_scale_enhancement (/root/reference/enhancers/multi_scale.py:17-60, :87-94):
//   for s in {1, 1/2, 1/4}:  img_s = bilinear(x, size=(int(H*s), int(W*s)), align_corners=False)
//       features_s = cat[img_s (3), luma .299/.587/.114 (1), sqrt(gx^2+gy^2) of torch.gradient per channel (3)]
//   gain = 1 + 0.1 * sum_s w_s * mean(features_s),   w = (0.5, 0.3, 0.2)
//
// The reference launches ~25 eager ops and re-reads the image ~10x.  Two paths here:
//   * streaming (H % 4 == 0 and W % 4 == 0, the named 1080p/4K shapes): ONE read of x.  At exact 1/2 and 1/4
//     scales torch's bilinear sample points fall on pixel-pair midpoints, so the 1/2 image is the 2x2 mean
//     and the 1/4 image is the mean of the centre 2x2 of every 4x4 block -- both fall out of the rows a warp
//     already holds in registers, and all 3 x 7 channel sums come out of that one pass (k_ms_stream).
//   * generic (any size, and whenever the feature maps themselves are requested): a bilinear down-sample
//     kernel followed by one feature kernel per scale.
// Sums are fp64 per thread -> warp shuffle -> one partial per CTA -> the last CTA of the image adds the
// partials in index order (deterministic) and writes the three means and the gain.
#include <algorithm>

#include "upr_maps.cuh"
#include <type_traits>

namespace upr {

constexpr int kMsThreads = 256;
constexpr int kMsMaxParts = 4096;

__device__ __forceinline__ double ms_block_sum(double v, double* s_red)
{
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) s_red[wid] = v;
    __syncthreads();
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < kMsThreads / 32; ++i) t += s_red[i];
    return t;
}

// torch.gradient along one axis (unit spacing, edge_order=1)
__device__ __forceinline__ float grad1(float m, float c, float p, int i, int len)
{
    if (len == 1) return 0.0f;
    if (i == 0) return __fsub_rn(p, c);
    if (i == len - 1) return __fsub_rn(c, m);
    return __fmul_rn(__fsub_rn(p, m), 0.5f);  // (p - m) / 2 : exact halving
}

template <bool kExactSqrt>
__device__ __forceinline__ float edge_mag(float gx, float gy)
{
    const float s = __fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy));
    if (kExactSqrt) return __fsqrt_rn(s);
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(s));
    return r;
}

__device__ __forceinline__ float luma601(float r, float g, float b)
{
    return __fadd_rn(__fadd_rn(__fmul_rn(0.299f, r), __fmul_rn(0.587f, g)), __fmul_rn(0.114f, b));
}

// means3 / gain from the three fp64 sums (multi_scale.py:90-94: fp32 .item() values accumulated in a Python float)
__device__ __forceinline__ void ms_finalize(const double sums[3], const double counts[3], float* means3, float* gain,
                                            double* gain64)
{
    const double wts[3] = {0.5, 0.3, 0.2};
    double factor = 1.0;
#pragma unroll
    for (int s = 0; s < 3; ++s) {
        const float m = float(sums[s] / (7.0 * counts[s]));
        means3[s] = m;
        factor += wts[s] * double(m) * 0.1;
    }
    *gain = float(factor);
    if (gain64) *gain64 = factor;
}

// -----------------------------------------------------------------------------------------
// generic path
// -----------------------------------------------------------------------------------------
// F.interpolate(mode='bilinear', align_corners=False, size=(oh, ow)) of [planes][h][w]
__global__ void __launch_bounds__(kMsThreads)
k_ms_downsample(const float* __restrict__ src, int h, int w, float* __restrict__ dst, int oh, int ow, long long planes)
{
    const float sy = __fdiv_rn(float(h), float(oh)), sx = __fdiv_rn(float(w), float(ow));
    const long long total = planes * oh * ow;
    const long long stride = (long long)gridDim.x * kMsThreads;
    for (long long it = (long long)blockIdx.x * kMsThreads + threadIdx.x; it < total; it += stride) {
        const long long pl = it / ((long long)oh * ow);
        const int rem = int(it - pl * oh * ow);
        const int y = rem / ow, x = rem - y * ow;
        float fy = __fsub_rn(__fmul_rn(__fadd_rn(float(y), 0.5f), sy), 0.5f);
        float fx = __fsub_rn(__fmul_rn(__fadd_rn(float(x), 0.5f), sx), 0.5f);
        fy = fy < 0.0f ? 0.0f : fy;
        fx = fx < 0.0f ? 0.0f : fx;
        const int y0 = int(fy), x0 = int(fx);
        const int y1 = y0 + (y0 < h - 1 ? 1 : 0), x1 = x0 + (x0 < w - 1 ? 1 : 0);
        const float ly = __fsub_rn(fy, float(y0)), hy = __fsub_rn(1.0f, ly);
        const float lx = __fsub_rn(fx, float(x0)), hx = __fsub_rn(1.0f, lx);
        const float* p = src + pl * (long long)h * w;
        const float a = __ldg(p + (long long)y0 * w + x0), b = __ldg(p + (long long)y0 * w + x1);
        const float c = __ldg(p + (long long)y1 * w + x0), d = __ldg(p + (long long)y1 * w + x1);
        const float top = __fadd_rn(__fmul_rn(hx, a), __fmul_rn(lx, b));
        const float bot = __fadd_rn(__fmul_rn(hx, c), __fmul_rn(lx, d));
        dst[it] = __fadd_rn(__fmul_rn(hy, top), __fmul_rn(ly, bot));
    }
}

// features of one scale: img [n][3][h][w] -> optional feat [n][7][h][w], partial sums [n][parts]
template <bool kWrite>
__global__ void __launch_bounds__(kMsThreads)
k_ms_features(const float* __restrict__ img, int h, int w, float* __restrict__ feat, double* __restrict__ partial)
{
    __shared__ double s_red[kMsThreads / 32];
    const int f = blockIdx.y, parts = gridDim.x;
    const long long plane = (long long)h * w;
    const float* base = img + (long long)f * 3 * plane;
    float* fo = kWrite ? feat + (long long)f * 7 * plane : nullptr;
    double acc = 0.0;
    const long long stride = (long long)parts * kMsThreads;
    for (long long it = (long long)blockIdx.x * kMsThreads + threadIdx.x; it < plane; it += stride) {
        const int y = int(it / w), x = int(it - (long long)y * w);
        float v[3], e[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float* p = base + c * plane + it;
            v[c] = __ldg(p);
            const float xm = x > 0 ? __ldg(p - 1) : 0.0f, xp = x < w - 1 ? __ldg(p + 1) : 0.0f;
            const float ym = y > 0 ? __ldg(p - w) : 0.0f, yp = y < h - 1 ? __ldg(p + w) : 0.0f;
            e[c] = edge_mag<true>(grad1(xm, v[c], xp, x, w), grad1(ym, v[c], yp, y, h));
        }
        const float lum = luma601(v[0], v[1], v[2]);
        if (kWrite) {
            fo[it] = v[0];
            fo[plane + it] = v[1];
            fo[2 * plane + it] = v[2];
            fo[3 * plane + it] = lum;
            fo[4 * plane + it] = e[0];
            fo[5 * plane + it] = e[1];
            fo[6 * plane + it] = e[2];
        }
        acc += double(v[0]) + double(v[1]) + double(v[2]) + double(lum) + double(e[0]) + double(e[1]) + double(e[2]);
    }
    acc = ms_block_sum(acc, s_red);
    if (threadIdx.x == 0) partial[(long long)f * parts + blockIdx.x] = acc;
}

// one thread per image: add the per-CTA partials of the three scales in index order
__global__ void k_ms_finalize(const double* __restrict__ p0, const double* __restrict__ p1, const double* __restrict__ p2,
                              int parts0, int parts1, int parts2, double c0, double c1, double c2, int n,
                              float* __restrict__ means, float* __restrict__ gain)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    double sums[3] = {0.0, 0.0, 0.0};
    for (int k = 0; k < parts0; ++k) sums[0] += p0[(long long)f * parts0 + k];
    for (int k = 0; k < parts1; ++k) sums[1] += p1[(long long)f * parts1 + k];
    for (int k = 0; k < parts2; ++k) sums[2] += p2[(long long)f * parts2 + k];
    const double counts[3] = {c0, c1, c2};
    ms_finalize(sums, counts, means + 3 * f, gain + f, nullptr);
}

// -----------------------------------------------------------------------------------------
// streaming path (H % 4 == 0, W % 4 == 0: the named shapes): one warp per (frame, 120-column band, row segment), no shared
// memory, no block barrier.  (A shared-memory tile kernel that staged a 72 x 40 halo tile and derived the half / quarter
// images from it ran 288 executed instructions per pixel at 80 % issue utilisation -- index arithmetic of three tile
// passes, 41 % halo re-staging, per-pixel luma and fp64 adds -- 1.31 ms against 0.36 ms on 16 x 4K; profiles/r2_multiscale_full.md.)
//   * a lane owns 4 full-resolution columns = 2 half-resolution columns = 1 quarter-resolution column and walks down
//     the segment one quarter row (4 image rows) at a time; the rows needed for vertical differences are carried in
//     registers, horizontal neighbours come from the adjacent lanes by shuffle (lanes 0 and 31 are halo);
//   * only what the means need is computed: sum(r+g+b+luma) is (1+w_c) * sum(channel c); the 2x2 block sums that give
//     the channel sums ARE the (unscaled) half-resolution pixels, the centre 2x2 of a 4x4 block the quarter pixel;
//     |grad| = 0.5 * sqrt(dx^2 + dy^2) with un-halved central differences (one-sided border differences doubled),
//     and the constant factors (0.5, 0.25) are applied once per step to the partial sums -- powers of two, so every
//     pixel value equals the reference's up to the approximate square root;
//   * fp32 partial sums per 16 pixels, fp64 across steps, ordered (deterministic) reduction by the last warp.
// Requires H % 4 == 0, W % 4 == 0, H/4 >= 2, W/4 >= 2 and 16-byte aligned rows.
// -----------------------------------------------------------------------------------------
constexpr int kMsBandCols = 120;

__device__ __forceinline__ float ms_mag(float dx, float dy)
{
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(__fmaf_rn(dx, dx, __fmul_rn(dy, dy))));
    return r;
}

// sum over the lane's pixels of sqrt(dx^2 + dy^2) for one row of 4 / 2 / 1 values; dy is already formed.
// Four-value rows: dy arrives as two packed pairs, dx^2 + dy^2 is two FMUL2 + two FFMA2, the four roots are summed as a pair.
__device__ __forceinline__ float ms_edge4(f32x2 v01, f32x2 v23, f32x2 dy01, f32x2 dy23, bool isL, bool isR)
{
    float v[4];
    upk2(v01, v[0], v[1]);
    upk2(v23, v[2], v[3]);
    const float left = __shfl_up_sync(0xffffffffu, v[3], 1), right = __shfl_down_sync(0xffffffffu, v[0], 1);
    const float d10 = __fsub_rn(v[1], v[0]), d32 = __fsub_rn(v[3], v[2]);
    const float dx0 = isL ? __fadd_rn(d10, d10) : __fsub_rn(v[1], left);
    const float dx3 = isR ? __fadd_rn(d32, d32) : __fsub_rn(right, v[2]);
    const f32x2 dxa = pk2(dx0, __fsub_rn(v[2], v[0])), dxb = pk2(__fsub_rn(v[3], v[1]), dx3);
    float m[4];
    upk2(fma2(dxa, dxa, mul2(dy01, dy01)), m[0], m[1]);
    upk2(fma2(dxb, dxb, mul2(dy23, dy23)), m[2], m[3]);
    float r[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r[i]) : "f"(m[i]));
    float lo, hi;
    upk2(add2(pk2(r[0], r[1]), pk2(r[2], r[3])), lo, hi);
    return __fadd_rn(lo, hi);
}
__device__ __forceinline__ float ms_edge2(const float v[2], const float dy[2], bool isL, bool isR)
{
    const float left = __shfl_up_sync(0xffffffffu, v[1], 1), right = __shfl_down_sync(0xffffffffu, v[0], 1);
    const float d = __fsub_rn(v[1], v[0]), d2 = __fadd_rn(d, d);
    const float dx0 = isL ? d2 : __fsub_rn(v[1], left);
    const float dx1 = isR ? d2 : __fsub_rn(right, v[0]);
    return __fadd_rn(ms_mag(dx0, dy[0]), ms_mag(dx1, dy[1]));
}
__device__ __forceinline__ float ms_edge1(float v, float dy, bool isL, bool isR)
{
    const float left = __shfl_up_sync(0xffffffffu, v, 1), right = __shfl_down_sync(0xffffffffu, v, 1);
    const float dr = __fsub_rn(right, v), dl = __fsub_rn(v, left);
    const float dx = isL ? __fadd_rn(dr, dr) : (isR ? __fadd_rn(dl, dl) : __fsub_rn(right, left));
    return ms_mag(dx, dy);
}

// History (16 x 4K): one general step body, 60 SASS instructions per pixel (27 % of them MOVs, 38 branches per step), 128 registers,
// issue 76 %, DRAM read 1.12x the frames: 0.348 ms (profiles/r4_ms_stream_full.md) -> branch-free interior step (42 instructions per
// pixel) + L2 prefetch two steps ahead: 0.318 ms -> odd segments walk upwards (DRAM read 1.004x the frames): 0.307 ms = 5.2 TB/s.
// 16 warps per SM (128 registers; the interior body alone would take 136): tighter bounds spill (20 / 24 warps: 0.374 / 0.498 ms on
// the round-1 body).
__global__ void __launch_bounds__(32, 16)
k_ms_stream(const float* __restrict__ x, int h, int w, int bands, int seg_rows, double* __restrict__ partial,
            unsigned* __restrict__ tickets, float* __restrict__ means, float* __restrict__ gain)
{
    const int lane = threadIdx.x;
    const int band = blockIdx.x % bands, seg = blockIdx.x / bands;
    const int f = blockIdx.y, parts = gridDim.x;
    // Odd segments work on the vertically FLIPPED frame (every statistic here is symmetric under a row flip: squared differences,
    // 2x2 / centre block sums on a 4-row grid), i.e. they walk their rows upwards: neighbouring segments start from a common
    // boundary at the same time and meet at the other one, so the 8 halo rows of a segment are in L2 when it reads them
    // (same idea as k_saliency_stream2).  seg_rows does not depend on the batch, so neither does a row's direction.
    const bool flip = seg & 1;
    int r0 = seg * seg_rows, r1 = min(r0 + seg_rows, h);
    if (r0 >= h) return;     // (never: segs = ceil(h / seg_rows))
    if (flip) { const int a = h - r1, b = h - r0; r0 = a; r1 = b; }
    const int q0 = r0 >> 2, q1 = r1 >> 2, Q = h >> 2;
    const int c0 = band * kMsBandCols - 4 + lane * 4;
    const bool counted = lane >= 1 && lane <= 30 && c0 < w;
    const bool isL = c0 == 0, isR = c0 + 4 == w;
    const int cl = min(max(c0, 0), w - 4);
    const long long plane = (long long)h * w;
    const float* img = x + (long long)f * 3 * plane + cl;

    // rows 4q-2 / 4q-1 of the previous step as packed column pairs {0,1}, {2,3}; half rows as pairs; quarter pixels as scalars
    f32x2 P2[3][2], P3[3][2], HB0[3], HB1[3];
    float Q1[3], Q2[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        P2[c][0] = P2[c][1] = P3[c][0] = P3[c][1] = HB0[c] = HB1[c] = 0ull;
        Q1[c] = Q2[c] = 0.0f;
    }
    double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0;

    float4 N[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) N[j] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    // row r of the (possibly flipped) frame: base + r * rstep
    const float* img0 = flip ? img + (long long)(h - 1) * w : img;
    const long long rstep = flip ? -(long long)w : (long long)w;
    auto load_rows = [&](int q, int c) {
        const float* p = img0 + c * plane + (long long)(4 * q) * rstep;
#pragma unroll
        for (int j = 0; j < 4; ++j) N[j] = __ldg(reinterpret_cast<const float4*>(p + (long long)j * rstep));
    };
    // One step = the four image rows 4q .. 4q+3.  kI (interior step: 2 <= q, q0 < q < min(q1, Q - 1)) turns every border condition
    // into a compile-time constant: the segment's inner loop then has no branches, no selects and none of the register copies
    // that merging the border paths costs (the general body ran 60 instructions per pixel, 27 % of them MOVs).
    auto step = [&](const int q, auto interior_tag) {
            constexpr bool kI = decltype(interior_tag)::value;
            const bool have = kI || q < Q;                 // image rows 4q .. 4q+3 exist
            const bool inner = kI || (q >= q0 && q < q1);  // their statistics belong to this segment
            const bool prev_in = kI || q > q0;             // rows 4q-1 / 2q-1 / q-1 belong to this segment
            float t0 = 0.0f, t1 = 0.0f, t2 = 0.0f;   // this step's contribution to the three scale totals
            {   // L2 prefetch of the four rows two steps ahead, all three channels; the register loads above run one (step, channel)
                // ahead.  Swept on 16 x 4K with the branch-free interior step and the bidirectional walk: one step ahead 0.318 ms,
                // two 0.307, three 0.314, four 0.376 (the slower general body of round 1 wanted one step: 0.363 against 0.367 / 0.379)
                const int qp = q + 2;
                if (qp <= q1 && qp < Q) {
#pragma unroll
                    for (int c = 0; c < 3; ++c)
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            asm volatile("prefetch.global.L2 [%0];" ::"l"(img0 + c * plane + (long long)(4 * qp + j) * rstep));
                }
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float wsum = c == 0 ? 1.299f : (c == 1 ? 1.587f : 1.114f);   // 1 + luma weight
                // software pipeline: the four rows of the NEXT (step, channel) are requested before this one is reduced
                // (ncu: 54 % of the stall samples of the un-pipelined kernel sat on the first use of these loads).
                // Row j of the step as the two natural column pairs of its 128-bit load: A[j] = {0,1}, B[j] = {2,3}
                // (packed fp32: differences, squares and block sums run two lanes per issue slot; the kernel is issue-bound).
                f32x2 A[4], B[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) { A[j] = pk2(N[j].x, N[j].y); B[j] = pk2(N[j].z, N[j].w); }
                if (c < 2) { if (have) load_rows(q, c + 1); }
                else if (kI || (q + 1 <= q1 && q + 1 < Q)) load_rows(q + 1, 0);
                // 2x2 block sums (= 4 x half-resolution pixels) and the centre 2x2 (= 4 x quarter-resolution pixel)
                float s0, s1, s2, s3;
                upk2(add2(A[0], A[1]), s0, s1);
                upk2(add2(B[0], B[1]), s2, s3);
                const f32x2 HBa = pk2(__fadd_rn(s0, s1), __fadd_rn(s2, s3));        // half row 2q
                upk2(add2(A[2], A[3]), s0, s1);
                upk2(add2(B[2], B[3]), s2, s3);
                const f32x2 HBb = pk2(__fadd_rn(s0, s1), __fadd_rn(s2, s3));        // half row 2q+1
                float c1lo, c1hi, c2lo, c2hi;
                upk2(add2(A[1], A[2]), c1lo, c1hi);      // rows 1+2, columns 0 | 1
                upk2(add2(B[1], B[2]), c2lo, c2hi);      // rows 1+2, columns 2 | 3
                const float Qc = __fadd_rn(c1hi, c2lo);
                float e0 = 0.0f, e1 = 0.0f, e2 = 0.0f;
                const f32x2 two = pk2(2.0f, 2.0f);
                // ---- rows completed by this step: image row 4q-1, half row 2q-1, quarter row q-1 ----
                if (kI || q >= 1) {
                    f32x2 dy4a, dy4b, dy2p;
                    if (have) {
                        dy4a = sub2(A[0], P2[c][0]); dy4b = sub2(B[0], P2[c][1]);
                        dy2p = sub2(HBa, HB0[c]);
                    } else {
                        dy4a = mul2(sub2(P3[c][0], P2[c][0]), two); dy4b = mul2(sub2(P3[c][1], P2[c][1]), two);
                        dy2p = mul2(sub2(HB1[c], HB0[c]), two);
                    }
                    float dy1;
                    if (!kI && q == 1) { const float d = __fsub_rn(Qc, Q1[c]); dy1 = __fadd_rn(d, d); }       // quarter row 0: one-sided
                    else if (have) dy1 = __fsub_rn(Qc, Q2[c]);
                    else { const float d = __fsub_rn(Q1[c], Q2[c]); dy1 = __fadd_rn(d, d); }          // last quarter row
                    const float a0 = ms_edge4(P3[c][0], P3[c][1], dy4a, dy4b, isL, isR);
                    float hv[2], hd[2];
                    upk2(HB1[c], hv[0], hv[1]);
                    upk2(dy2p, hd[0], hd[1]);
                    const float a1 = ms_edge2(hv, hd, isL, isR);
                    const float a2 = ms_edge1(Q1[c], dy1, isL, isR);
                    if (prev_in) { e0 = a0; e1 = a1; e2 = a2; }
                }
                // ---- rows 4q .. 4q+2, half row 2q ----
                if (have) {
                    f32x2 dyAa, dyAb, dyHp;
                    if (!kI && q == 0) {
                        dyAa = mul2(sub2(A[1], A[0]), two); dyAb = mul2(sub2(B[1], B[0]), two);
                        dyHp = mul2(sub2(HBb, HBa), two);
                    } else {
                        dyAa = sub2(A[1], P3[c][0]); dyAb = sub2(B[1], P3[c][1]);
                        dyHp = sub2(HBb, HB1[c]);
                    }
                    const float a0 = __fadd_rn(__fadd_rn(ms_edge4(A[0], B[0], dyAa, dyAb, isL, isR),
                                                         ms_edge4(A[1], B[1], sub2(A[2], A[0]), sub2(B[2], B[0]), isL, isR)),
                                               ms_edge4(A[2], B[2], sub2(A[3], A[1]), sub2(B[3], B[1]), isL, isR));
                    float hv[2], hd[2];
                    upk2(HBa, hv[0], hv[1]);
                    upk2(dyHp, hd[0], hd[1]);
                    const float a1 = ms_edge2(hv, hd, isL, isR);
                    if (inner) {
                        e0 = __fadd_rn(e0, a0);
                        e1 = __fadd_rn(e1, a1);
                        float f0, f1;
                        upk2(add2(HBa, HBb), f0, f1);
                        const float sfull = __fadd_rn(f0, f1);
                        // channel sums: full = sum of the 16 pixels, half = 0.25 * the same, quarter = 0.25 * centre sum
                        t0 = __fmaf_rn(wsum, sfull, t0);
                        t1 = __fmaf_rn(wsum * 0.25f, sfull, t1);
                        t2 = __fmaf_rn(wsum * 0.25f, Qc, t2);
                    }
                    P2[c][0] = A[2]; P2[c][1] = B[2]; P3[c][0] = A[3]; P3[c][1] = B[3];
                    HB0[c] = HBa; HB1[c] = HBb;
                    Q2[c] = Q1[c]; Q1[c] = Qc;
                }
                // |grad| = 0.5 * sqrt(.) of un-halved differences; half / quarter pixels carry their factor 0.25
                t0 = __fmaf_rn(0.5f, e0, t0);
                t1 = __fmaf_rn(0.125f, e1, t1);
                t2 = __fmaf_rn(0.125f, e2, t2);
            }
            if (counted) { acc0 += double(t0); acc1 += double(t1); acc2 += double(t2); }
    };
    if (r0 < h) {
        const int qs = max(q0 - 1, 0);
        const int qi0 = max(max(q0 + 1, 2), qs), qi1 = min(q1, Q - 1);
        if (qs < Q) load_rows(qs, 0);
#pragma unroll 1
        for (int q = qs; q <= q1; ++q) {
            if (q == qi0) {
#pragma unroll 1
                for (; q < qi1; ++q) step(q, std::true_type{});
            }
            step(q, std::false_type{});
        }
    }
    acc0 = warp_sum(acc0);
    acc1 = warp_sum(acc1);
    acc2 = warp_sum(acc2);
    double* pp = partial + ((long long)f * parts + blockIdx.x) * 3;
    int last = 0;
    if (lane == 0) {
        pp[0] = acc0; pp[1] = acc1; pp[2] = acc2;
        __threadfence();
        const unsigned t = atomicAdd(tickets + f, 1u);
        last = (t == unsigned(parts - 1));
        if (last) tickets[f] = 0;
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (!last) return;
    __threadfence();
    // last warp of the frame: ordered sum of the partials (lane-strided, then a fixed shuffle tree)
    double sums[3] = {0.0, 0.0, 0.0};
    for (int k = lane; k < parts; k += 32) {
        const double* qd = partial + ((long long)f * parts + k) * 3;
        sums[0] += __ldcg(qd);
        sums[1] += __ldcg(qd + 1);
        sums[2] += __ldcg(qd + 2);
    }
    sums[0] = warp_sum(sums[0]);
    sums[1] = warp_sum(sums[1]);
    sums[2] = warp_sum(sums[2]);
    if (lane == 0) {
        const double counts[3] = {double(h) * w, double(h / 2) * (w / 2), double(h / 4) * (w / 4)};
        ms_finalize(sums, counts, means + 3 * f, gain + f, nullptr);
    }
}

struct MsLayout {
    size_t off_partial, off_tickets, off_half, off_quar, total;
    int oh2, ow2, oh4, ow4;
};

static MsLayout ms_layout(int n, int h, int w)
{
    // tickets first, at an offset that does not depend on (n, h, w): the kernels leave them at zero, so a workspace that was
    // zero-filled once can be reused for any later batch size or shape (with the tickets behind the n-dependent partial sums a
    // call with another n found stale data where it expected clean tickets -- caught by the 2 x 1080p oracle test)
    MsLayout L;
    L.oh2 = int(h * 0.5); L.ow2 = int(w * 0.5); L.oh4 = int(h * 0.25); L.ow4 = int(w * 0.25);
    L.off_tickets = 0;
    L.off_partial = align_up(size_t(65536) * sizeof(unsigned), 256);
    L.off_half = align_up(L.off_partial + size_t(n) * kMsMaxParts * 3 * sizeof(double), 256);
    L.off_quar = align_up(L.off_half + size_t(n) * 3 * L.oh2 * L.ow2 * sizeof(float), 256);
    L.total = align_up(L.off_quar + size_t(n) * 3 * L.oh4 * L.ow4 * sizeof(float), 256);
    return L;
}

static int ms_parts(int n, long long px)
{
    const long long by_work = std::max<long long>(1, px / (kMsThreads * 4));
    const long long by_fill = (4LL * kNumSMsB200 + n - 1) / n;
    return int(std::max<long long>(1, std::min<long long>(std::min(by_work, by_fill), kMsMaxParts)));
}

bool ms_stream_geometry(int h, int w, const float* x, MsStreamGeom* geo)
{
    if (!(h % 4 == 0 && w % 4 == 0 && h / 4 >= 2 && w / 4 >= 2 && aligned16(x))) return false;
    // one warp per (band, row segment, frame)
    const int bands = (w + kMsBandCols - 1) / kMsBandCols;
    // 64-row segments whatever the batch: odd segments walk upwards, and the direction of a row must not depend on nf
    // (96 / 128 / 192 / 256 rows: 0.300 / 0.302 / 0.331 / 0.324 ms against 0.308 ms per 16 x 4K -- fewer general border steps, fewer warps)
    int seg_rows = 64;
    // (very wide frames: longer segments keep the per-frame partial count inside the workspace)
    while ((long long)bands * ((h + seg_rows - 1) / seg_rows) > kMsMaxParts && seg_rows < h) seg_rows *= 2;
    if ((long long)bands * ((h + seg_rows - 1) / seg_rows) > kMsMaxParts) return false;
    *geo = MsStreamGeom{bands, seg_rows};
    return true;
}

int ms_stream_launch_range(const float* x, int nf, int h, int w, const MsStreamGeom& geo, void* ms_ws, size_t ms_ws_bytes,
                           int n_total, int f0, float* means3, float* gain, cudaStream_t s)
{
    if (nf <= 0 || f0 < 0 || f0 + nf > n_total || n_total > 65535 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    if (!x || !ms_ws || !means3 || !gain) return UPR_E_NULL;
    const MsLayout lay = ms_layout(n_total, h, w);
    if (ms_ws_bytes < lay.total || (reinterpret_cast<uintptr_t>(ms_ws) & 255u)) return UPR_E_WORKSPACE;
    auto* base = static_cast<unsigned char*>(ms_ws);
    auto* partial = reinterpret_cast<double*>(base + lay.off_partial) + size_t(f0) * kMsMaxParts * 3;
    auto* tickets = reinterpret_cast<unsigned*>(base + lay.off_tickets) + f0;
    const int segs = (h + geo.seg_rows - 1) / geo.seg_rows;
    k_ms_stream<<<dim3(geo.bands * segs, nf), 32, 0, s>>>(x, h, w, geo.bands, geo.seg_rows, partial, tickets, means3, gain);
    UPR_LAUNCH_CHECK();
    return UPR_OK;
}

static int ms_run(const float* x, int n, int h, int w, float* means, float* gain, float* f1, float* f2, float* f3,
                  void* ws, size_t ws_bytes, cudaStream_t s, bool allow_fused)
{
    if (n < 0 || n > 65535 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    const MsLayout lay = ms_layout(std::max(n, 1), h, w);
    if (lay.oh4 < 1 || lay.ow4 < 1) return UPR_E_SHAPE;  // torch raises on a zero-sized interpolate target
    if (n == 0) return UPR_OK;
    if (!x || !ws) return UPR_E_NULL;
    if (ws_bytes < lay.total || (reinterpret_cast<uintptr_t>(ws) & 255u)) return UPR_E_WORKSPACE;
    auto* base = static_cast<unsigned char*>(ws);
    auto* partial = reinterpret_cast<double*>(base + lay.off_partial);
    auto* tickets = reinterpret_cast<unsigned*>(base + lay.off_tickets);
    auto* half = reinterpret_cast<float*>(base + lay.off_half);
    auto* quar = reinterpret_cast<float*>(base + lay.off_quar);
    const bool want_feat = f1 || f2 || f3;
    if (want_feat && !(f1 && f2 && f3)) return UPR_E_NULL;
    if (!want_feat && (!means || !gain)) return UPR_E_NULL;

    MsStreamGeom geo{};
    if (allow_fused && !want_feat && ms_stream_geometry(h, w, x, &geo))
        return ms_stream_launch_range(x, n, h, w, geo, ws, ws_bytes, n, 0, means, gain, s);
    // generic: down-sample, then one feature kernel per scale
    {
        const long long t2 = (long long)n * 3 * lay.oh2 * lay.ow2, t4 = (long long)n * 3 * lay.oh4 * lay.ow4;
        const int g2 = int(std::min<long long>((t2 + kMsThreads - 1) / kMsThreads, 8LL * kNumSMsB200));
        const int g4 = int(std::min<long long>((t4 + kMsThreads - 1) / kMsThreads, 8LL * kNumSMsB200));
        k_ms_downsample<<<g2, kMsThreads, 0, s>>>(x, h, w, half, lay.oh2, lay.ow2, (long long)n * 3);
        UPR_LAUNCH_CHECK();
        k_ms_downsample<<<g4, kMsThreads, 0, s>>>(x, h, w, quar, lay.oh4, lay.ow4, (long long)n * 3);
        UPR_LAUNCH_CHECK();
    }
    const int p0 = ms_parts(n, (long long)h * w), p1 = ms_parts(n, (long long)lay.oh2 * lay.ow2),
              p2 = ms_parts(n, (long long)lay.oh4 * lay.ow4);
    double* pp0 = partial;
    double* pp1 = pp0 + (size_t)n * p0;
    double* pp2 = pp1 + (size_t)n * p1;
    if (want_feat) {
        k_ms_features<true><<<dim3(p0, n), kMsThreads, 0, s>>>(x, h, w, f1, pp0);
        k_ms_features<true><<<dim3(p1, n), kMsThreads, 0, s>>>(half, lay.oh2, lay.ow2, f2, pp1);
        k_ms_features<true><<<dim3(p2, n), kMsThreads, 0, s>>>(quar, lay.oh4, lay.ow4, f3, pp2);
    } else {
        k_ms_features<false><<<dim3(p0, n), kMsThreads, 0, s>>>(x, h, w, nullptr, pp0);
        k_ms_features<false><<<dim3(p1, n), kMsThreads, 0, s>>>(half, lay.oh2, lay.ow2, nullptr, pp1);
        k_ms_features<false><<<dim3(p2, n), kMsThreads, 0, s>>>(quar, lay.oh4, lay.ow4, nullptr, pp2);
    }
    UPR_LAUNCH_CHECK();
    if (means && gain) {
        k_ms_finalize<<<(n + 63) / 64, 64, 0, s>>>(pp0, pp1, pp2, p0, p1, p2, double(h) * w, double(lay.oh2) * lay.ow2,
                                                    double(lay.oh4) * lay.ow4, n, means, gain);
        UPR_LAUNCH_CHECK();
    }
    return UPR_OK;
}

// upr_retinex_multiscale_typed_*: the schedule of upr_multiscale_enhance_f32 with the map epilogue in place of the gain pass
static int ms_maps_run(const MapsArgs& m, float* means, float* gain, int n, int h, int w, void* ws, size_t ws_bytes, cudaStream_t s)
{
    if (n < 0 || n > 65535 || h <= 0 || w <= 0 || int(h * 0.25) < 1 || int(w * 0.25) < 1) return UPR_E_SHAPE;
    bool done;
    const int rc = maps_check(m, n, &done);
    if (done) return rc;
    if (!means || !gain || !ws) return UPR_E_NULL;
    MsStreamGeom geo{};
    if (!ms_stream_geometry(h, w, m.x, &geo)) {
        const int rs = ms_run(m.x, n, h, w, means, gain, nullptr, nullptr, nullptr, ws, ws_bytes, s, true);
        if (rs) return rs;
        return maps_epilogue(m, n, h, w, FrameGain{gain}, s);
    }
    const long long plane = (long long)h * w;
    return run_chunked(s, n, chunk_frames(plane), [&](int f0, int nf, cudaStream_t cs) {
        const int rs = ms_stream_launch_range(m.x + f0 * 3 * plane, nf, h, w, geo, ws, ws_bytes, n, f0, means + 3 * f0, gain + f0, cs);
        if (rs) return rs;
        return maps_epilogue(m.at(f0, plane), nf, h, w, FrameGain{gain + f0}, cs);
    });
}

}  // namespace upr

extern "C" {

int upr_retinex_multiscale_typed_f32(const float* x_nchw, const void* illu_n1hw, int illu_dtype, const void* e_nchw, int e_dtype,
                                     int flags, float* out_nchw, float* means_n_by_3, float* gain_per_image, int n, int h, int w,
                                     float eps, void* workspace, size_t workspace_bytes, upr_stream_t stream)
{
    const upr::MapsArgs m{x_nchw, illu_n1hw, illu_dtype, e_nchw, e_dtype, flags, eps, out_nchw, nullptr, nullptr};
    return upr::ms_maps_run(m, means_n_by_3, gain_per_image, n, h, w, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int upr_retinex_multiscale_typed_u8(const float* x_nchw, const void* illu_n1hw, int illu_dtype, const void* e_nchw, int e_dtype,
                                    int flags, unsigned char* out_nhwc, unsigned char* illu_nhw1, float* means_n_by_3,
                                    float* gain_per_image, int n, int h, int w, float eps, void* workspace, size_t workspace_bytes,
                                    upr_stream_t stream)
{
    const upr::MapsArgs m{x_nchw, illu_n1hw, illu_dtype, e_nchw, e_dtype, flags, eps, nullptr, out_nhwc, illu_nhw1};
    return upr::ms_maps_run(m, means_n_by_3, gain_per_image, n, h, w, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

size_t upr_multiscale_workspace_bytes(int n, int h, int w)
{
    if (n < 0 || h <= 0 || w <= 0) return 0;
    return upr::ms_layout(std::max(n, 1), h, w).total;
}

int upr_multiscale_stats_f32(const float* x_nchw, int n, int h, int w, float* means_n_by_3, float* gain_per_image,
                             void* workspace, size_t workspace_bytes, int flags, upr_stream_t stream)
{
    return upr::ms_run(x_nchw, n, h, w, means_n_by_3, gain_per_image, nullptr, nullptr, nullptr, workspace,
                       workspace_bytes, static_cast<cudaStream_t>(stream), (flags & 1) == 0);
}

int upr_multiscale_features_f32(const float* x_nchw, int n, int h, int w, float* feat_full, float* feat_half,
                                float* feat_quarter, float* means_n_by_3, float* gain_per_image, void* workspace,
                                size_t workspace_bytes, upr_stream_t stream)
{
    if (!feat_full || !feat_half || !feat_quarter) return UPR_E_NULL;
    return upr::ms_run(x_nchw, n, h, w, means_n_by_3, gain_per_image, feat_full, feat_half, feat_quarter, workspace,
                       workspace_bytes, static_cast<cudaStream_t>(stream), false);
}

int upr_multiscale_enhance_f32(const float* x_nchw, const float* enh_nchw, float* out_nchw, float* means_n_by_3, float* gain_per_image,
                               int n, int h, int w, void* workspace, size_t workspace_bytes, upr_stream_t stream)
{
    using namespace upr;
    if (n < 0 || n > 65535 || h <= 0 || w <= 0) return UPR_E_SHAPE;
    if (n == 0) return UPR_OK;
    if (!x_nchw || !enh_nchw || !out_nchw || !means_n_by_3 || !gain_per_image || !workspace) return UPR_E_NULL;
    auto s = static_cast<cudaStream_t>(stream);
    MsStreamGeom geo{};
    if (!ms_stream_geometry(h, w, x_nchw, &geo)) {
        const int rc = upr_multiscale_stats_f32(x_nchw, n, h, w, means_n_by_3, gain_per_image, workspace, workspace_bytes, 0, stream);
        if (rc) return rc;
        return scale_clamp_launch(enh_nchw, gain_per_image, out_nchw, n, 3, h, w, s);
    }
    // Chunks of ~25 Mpx, statistics then gain pass of a chunk on one of two side streams: the latency-bound statistics kernel of
    // chunk i + 1 runs under the bandwidth-bound gain pass of chunk i (16 x 4K: 0.82 ms back to back -> 0.79 ms; the frames are
    // independent, so the results do not depend on the schedule).
    const long long plane = (long long)h * w;
    return run_chunked(s, n, chunk_frames(plane), [&](int f0, int nf, cudaStream_t cs) {
        const int rc = ms_stream_launch_range(x_nchw + f0 * 3 * plane, nf, h, w, geo, workspace, workspace_bytes, n, f0,
                                              means_n_by_3 + 3 * f0, gain_per_image + f0, cs);
        if (rc) return rc;
        return scale_clamp_launch(enh_nchw + f0 * 3 * plane, gain_per_image + f0, out_nchw + f0 * 3 * plane, nf, 3, h, w, cs);
    });
}

}  // extern "C"
