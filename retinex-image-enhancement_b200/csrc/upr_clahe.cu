// upr_clahe.cu -- CLAHE-in-Lab for sm_100a (B200).
//
// Replaces AdaptiveParameterAdjuster.apply_clahe_enhancement
// (/root/reference/enhancers/adaptive_params.py:121-169), i.e. the host chain
//   (x*255).astype(u8) -> RGB2BGR -> BGR2LAB -> split -> CLAHE(2.0,(8,8)).apply(L) -> merge
//   -> LAB2BGR -> BGR2RGB -> /255
// with two kernels per batch and a 3 B/px u8 Lab intermediate:
//
//   K1  k_hist_lab_vec3  one CTA per (frame, tile, row-strip): planar f32 RGB -> u8 quantise -> OpenCV fixed-point
//                        Lab; stores L,a,b (u8 planes); per-THREAD private byte counters in shared memory build the
//                        tile histogram without atomics; the CTA (or the last strip CTA of the tile) then does
//                        clip -> redistribute -> prefix scan -> LUT in place.
//   K3  k_map_vec5       persistent CTAs pulling (frame, interpolation cell, row-strip) items: the four tile LUTs
//                        that surround a cell are interleaved into one 32-bit word per grey level, so the bilinear
//                        LUT interpolation costs ONE shared-memory lookup per pixel; fused with Lab -> sRGB (integer
//                        path) and the /255 de-quantisation.
//   (k_*_generic handle ragged shapes incl. OpenCV's padding quirk; the retired kernel generations and what each change
//    bought are recorded in profiles/r2_clahe.md and profiles/r3_clahe.md.)
//
// All fixed-point recipes follow SURVEY.md Appendix A (pinned against the cv2 binary by the
// oracle tests).  fp32 products/sums of the interpolation use __fmul_rn/__fadd_rn so that ptxas
// cannot contract them into FMAs: OpenCV evaluates them separately rounded (SURVEY finding 9).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "upr_common.cuh"
#include "upr_maps.cuh"
#include "upr_tables_gen.h"

namespace upr {

// ---------------------------------------------------------------------------------------------
// constant tables (device copies live in global memory; kernels stage what they need in smem)
// ---------------------------------------------------------------------------------------------
__device__ const uint16_t d_gamma[UPR_TAB_GAMMA_LEN] = UPR_TAB_GAMMA_INIT;
__device__ const uint16_t d_cbrt[UPR_TAB_CBRT_LEN] = UPR_TAB_CBRT_INIT;
__device__ const uint32_t d_labyf[UPR_TAB_LABYF_LEN] = UPR_TAB_LABYF_INIT;
__device__ const uint32_t d_outf_bits[UPR_TAB_INVGAMMA_F32BITS_LEN] = UPR_TAB_INVGAMMA_F32BITS_INIT;
__device__ __align__(16) const int16_t d_xzlin[UPR_TAB_XZLIN_LEN + 8] = UPR_TAB_XZLIN_INIT;   // padded to a multiple of 16 bytes
__device__ __align__(16) const uint8_t d_invgamma[UPR_TAB_INVGAMMA_LEN] = UPR_TAB_INVGAMMA_INIT;  // u8 outputs (packed u8 frames)

static const uint16_t h_gamma[UPR_TAB_GAMMA_LEN] = UPR_TAB_GAMMA_INIT;
static const uint16_t h_cbrt[UPR_TAB_CBRT_LEN] = UPR_TAB_CBRT_INIT;
static const uint32_t h_labyf[UPR_TAB_LABYF_LEN] = UPR_TAB_LABYF_INIT;
static const uint8_t h_invgamma[UPR_TAB_INVGAMMA_LEN] = UPR_TAB_INVGAMMA_INIT;

constexpr int kMaxTiles = 16;  // per axis, fast path; larger grids take the generic path
constexpr int kK1Threads = 256;
constexpr int kK3Threads = 256;

struct ClaheGeom {
    int n, h, w;
    int tiles_x, tiles_y;
    int tw, th;        // tile size in the (possibly padded) image
    int clip;          // integer clip limit, 0 = no clipping
    float lut_scale;   // 255 / (tw*th)
    int nstrips;       // K1 row strips per tile
    int strip_rows;
    uint32_t gam_bias; // 0 - 4 * 0x4B000000, passed as a PARAMETER: ptxas splits a compile-time constant off the gamma
                       // table address again and re-adds it per gather (one extra instruction per table lookup)
};

struct MapGeom {
    int n, h, w;
    int tiles_x, tiles_y;
    float inv_tw, inv_th;
    int nstrips;
    uint32_t ay_bias;  // 0 - 0x4B400000 * 128 as a parameter (see ClaheGeom::gam_bias)
    int bx[kMaxTiles + 2];  // cell c covers x in [bx[c], bx[c+1]); raw tile index of the cell is c-1
    int by[kMaxTiles + 2];
    // work-queue order of the persistent map kernel: LARGEST cells first.  Interior cells are a whole tile, border cells half of
    // one, corner cells a quarter; with the small ones at the very end of the queue the CTAs run dry within a quarter-item of
    // each other instead of a whole one.  order[] lists the cells by descending area in three size classes of n_class[] cells.
    int n_class[3];
    unsigned short order[(kMaxTiles + 1) * (kMaxTiles + 1)];
};

// queue position -> (frame, cell, strip): all frames' class-0 items, then all class-1 items, then all class-2 items
__device__ __forceinline__ void map_item(const MapGeom& g, int item, int& f, int& cell, int& strip)
{
    int base_rank = 0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int per = g.n_class[c] * g.nstrips;        // items of this class per frame
        const int all = per * g.n;
        if (item < all || c == 2) {
            f = item / max(per, 1);
            const int r = item - f * per;
            const int k = r / g.nstrips;
            strip = r - k * g.nstrips;
            cell = g.order[base_rank + k];
            return;
        }
        item -= all;
        base_rank += g.n_class[c];
    }
}

// ---------------------------------------------------------------------------------------------
// raw shared/global access helpers of the second-generation kernels
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_nc_u32(const uint8_t* p)
{
    uint32_t v;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_cs_f4(float* p, float a, float b, float c, float d)
{
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// Pipe budget notes (ncu, profiles/r1_clahe_full.md): the first-generation kernel was bound by the 16-lane ALU
// pipe (72 % busy: SHF/LOP3/LEA/IADD3/PRMT/VIMNMX/ISETP) while the FMA pipe idled at 36 % and the conversion
// pipe at 1 %.  Hence: table records with a 12-byte stride (address = index*12 + base is an IMAD, not a LEA),
// unpacked {quad, A, y} records (no LOP/SHF to split a packed word), all four LUT bytes converted by I2F.U8,
// shift+add pairs expressed so that they become one LEA.HI.SX32, and IMAD.WIDE global addressing.
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr)
{
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ int lds_s32_off(uint32_t addr, int off)
{
    int v;
    if (off == 4) asm("ld.shared.s32 %0, [%1+4];" : "=r"(v) : "r"(addr));
    else asm("ld.shared.s32 %0, [%1+8];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ float lds_f32(uint32_t addr)
{
    float v;
    asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
// base + idx*scale as ONE IMAD.WIDE on the FMA pipe.  `scale` is a run-time register (4 or 16 plus blockIdx.z == 0):
// with an immediate power of two ptxas lowers the same PTX to LEA + LEA.HI.X, two instructions on the ALU pipe,
// which is the pipe these kernels saturate.
__device__ __forceinline__ const void* wide_addr(const void* base, uint32_t idx, uint32_t scale)
{
    unsigned long long r;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(r) : "r"(idx), "r"(scale), "l"(base));
    return reinterpret_cast<const void*>(r);
}

// ---------------------------------------------------------------------------------------------
// device arithmetic (Appendix A.1 / A.2)
// ---------------------------------------------------------------------------------------------
// sRGB u8 -> Lab u8.  No clamps: over the whole 2^24 cube L is 0..255, a 42..226, b 20..223.
__device__ __forceinline__ void rgb_to_lab(int qr, int qg, int qb, const uint16_t* s_gamma, const uint16_t* s_cbrt,
                                           int& L, int& a, int& b)
{
    const int R = s_gamma[qr], G = s_gamma[qg], B = s_gamma[qb];
    const int fX = s_cbrt[(1777 * R + 1541 * G + 778 * B + 2048) >> 12];
    const int fY = s_cbrt[(871 * R + 2929 * G + 296 * B + 2048) >> 12];
    const int fZ = s_cbrt[(73 * R + 448 * G + 3575 * B + 2048) >> 12];
    L = (296 * fY - 1336934 + 16384) >> 15;
    a = (500 * (fX - fY) + 128 * 32768 + 16384) >> 15;
    b = (200 * (fY - fZ) + 128 * 32768 + 16384) >> 15;
}

__device__ __forceinline__ int rgb_to_l_only(int qr, int qg, int qb, const uint16_t* s_gamma, const uint16_t* s_cbrt)
{
    const int R = s_gamma[qr], G = s_gamma[qg], B = s_gamma[qb];
    const int fY = s_cbrt[(871 * R + 2929 * G + 296 * B + 2048) >> 12];
    return (296 * fY - 1336934 + 16384) >> 15;
}

__device__ __forceinline__ int ab_to_xz(int i)
{
    const int lin = i * 108 / 841 - 290;            // C truncating division (i may be negative)
    const int cub = (((i * i) >> 14) * i) >> 14;    // only selected for i > 3390 (all positive)
    return i <= 3390 ? lin : cub;
}

// Lab u8 -> three de-quantised f32 channels (s_outf[c] = float(invgamma[c]) / 255.f).
__device__ __forceinline__ void lab_to_rgb_f32(int L, int a, int b, const uint32_t* s_yf, const float* s_outf,
                                               float& r, float& g, float& bl)
{
    const uint32_t yf = s_yf[L];
    const int ify = int(yf & 0xffffu), y = int(yf >> 16);
    const int adiv = ((a * 268435 + 128) >> 13) - 4194;   // 5*53687 = 268435
    const int bdiv = ((b * 41943 + 16) >> 9) - 10484;
    const int x = ab_to_xz(ify + adiv);
    const int z = ab_to_xz(ify - bdiv);
    int ro = (12615 * x - 6296 * y - 2223 * z + 8192) >> 14;
    int go = (-3773 * x + 7684 * y + 185 * z + 8192) >> 14;
    int bo = (217 * x - 836 * y + 4715 * z + 8192) >> 14;
    ro = min(max(ro, 0), 4095);
    go = min(max(go, 0), 4095);
    bo = min(max(bo, 0), 4095);
    r = s_outf[ro];
    g = s_outf[go];
    bl = s_outf[bo];
}

// clip -> redistribute -> inclusive scan -> LUT, for one tile; blockDim.x must be 256, thread i
// owns bin i (Appendix A.3 steps 3-4).  s_tmp: >= 8 ints of shared scratch.
__device__ __forceinline__ void tile_lut_256(int hbin, int clip, float lut_scale, uint8_t* __restrict__ lut_out, int* s_tmp)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (clip > 0) {
        const int excess = max(hbin - clip, 0);
        hbin = min(hbin, clip);
        const int ws = warp_sum(excess);
        if (lane == 0) s_tmp[wid] = ws;
        __syncthreads();
        int clipped = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) clipped += s_tmp[i];
        __syncthreads();
        const int batch = clipped >> 8;
        const int resid = clipped & 255;
        hbin += batch;
        if (resid != 0) {
            const int step = max(256 / resid, 1);
            if (tid % step == 0 && tid / step < resid) ++hbin;
        }
    }
    int v = hbin;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    if (lane == 31) s_tmp[wid] = v;
    __syncthreads();
    int base = 0;
    for (int i = 0; i < wid; ++i) base += s_tmp[i];
    const int sum = v + base;
    const int r = __float2int_rn(__fmul_rn(__int2float_rn(sum), lut_scale));
    lut_out[tid] = uint8_t(min(max(r, 0), 255));
}

// Publishes a CTA's partial tile histogram; returns true (block-uniform) if this CTA must build
// the LUT, with `total` holding the complete histogram bin of thread `tid`.
__device__ __forceinline__ bool publish_hist(int& total, int32_t* __restrict__ hg, unsigned* __restrict__ ticket,
                                             int nparts, int* s_flag)
{
    const int tid = threadIdx.x;
    if (nparts == 1) {
        hg[tid] = total;
        return true;
    }
    atomicAdd(&hg[tid], total);
    __threadfence();
    __syncthreads();
    if (tid == 0) *s_flag = (atomicAdd(ticket, 1u) == unsigned(nparts - 1));
    __syncthreads();
    if (!*s_flag) return false;
    __threadfence();
    total = __ldcg(&hg[tid]);
    return true;
}

// ---------------------------------------------------------------------------------------------
// K1 fast path (W % tiles_x == 0, H % tiles_y == 0, tile width % 4 == 0, 16-byte aligned planes): per-pixel arithmetic.
// The first version ran 80 SASS instructions per pixel at 64 % issue utilisation; this is the "instruction diet" that
// replaced it.  Same arithmetic as Appendix A.1, hence bit-identical Lab planes / histograms / LUTs:
//   * quantisation on the FMA pipe: for 0 <= x <= 1 (checked once per 12 values with three-input integer maxima on
//     the raw bit patterns) trunc(x*255) is the low mantissa of  RZ(x*255 + 2^23);  those bits times four plus a
//     constant IS the shared address of the gamma entry.  Anything else (negative, > 1, NaN, inf) takes the exact
//     general path (numpy's wrap-around semantics, see quantize_u8);
//   * the gamma table is stored as fp32 and the three 3x3 dot products run as FFMA chains (every partial sum is an
//     integer < 2^24, hence exact); floor(S / 4096) falls out of one more FFMA.RZ against 2^23, again as address bits;
//   * L, a, b are produced pre-scaled so that the result sits in byte 2 of a register: one PRMT assembles a Lab word,
//     no shifts, no masks;
//   * the private-counter address ((L >> 2) << 10 | (L & 3)) is (L * 257) & 0xFC03: one PRMT, one LOP3 (which also ORs
//     in the thread's column); the counter is bumped by ONE red.shared.add.u32.
// ---------------------------------------------------------------------------------------------
// hides a value's provenance from ptxas (otherwise `bits*4 + (base - K)` is re-associated into two adds per use)
__device__ __forceinline__ uint32_t opaque(uint32_t x)
{
    uint32_t y;
    asm volatile("mov.b32 %0, %1;" : "=r"(y) : "r"(x));
    return y;
}
// base + idx * K (K an immediate) as ONE IMAD.WIDE.U32 with a 64-bit addend: nothing 64-bit to keep live but the base
template <uint32_t K>
__device__ __forceinline__ const char* wide_imm(const char* base, uint32_t idx)
{
    unsigned long long r;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(r) : "r"(idx), "n"(K), "l"(base));
    return reinterpret_cast<const char*>(r);
}

template <typename T>
__device__ __forceinline__ T* opaque_ptr(T* p)
{
    unsigned long long v = reinterpret_cast<unsigned long long>(p);
    asm volatile("mov.b64 %0, %0;" : "+l"(v));
    return reinterpret_cast<T*>(v);
}

__device__ __forceinline__ void prefetch_l2(const void* p)
{
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}
__device__ __forceinline__ void st_global_u32(const void* p, uint32_t v)
{
    // no "memory" clobber: the Lab words are never read back by the storing kernel, and a clobber would pin every
    // shared-memory access of the surrounding code in program order
    asm volatile("st.global.u32 [%0], %1;" ::"l"(p), "r"(v));
}
__device__ __forceinline__ float4 ld_nc_f4(const void* p)
{
    float4 v;
    asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ uint32_t ld_nc_u32p(const void* p)
{
    uint32_t v;
    asm("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr)
{
    uint32_t v;
    asm("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

struct K1Tables {
    uint32_t gam_q;    // &s_gammaf[0] - 4 * 0x4B000000: address of gamma[q] from the magic-add bits of q
    uint32_t gam;      // &s_gammaf[0]
    uint32_t cbr_q;    // &s_cbrt[0] - 2 * 0x4B000000
    uint32_t four, sixteen;
};

__device__ __forceinline__ void k1_core(const float (&R)[4], const float (&G)[4], const float (&B)[4], const K1Tables& t,
                                        unsigned char* s_cnt, uint32_t tid4, uint32_t& wl, uint32_t& wa, uint32_t& wb);

// 12 floats (4 px x RGB) -> three Lab words + four counter increments
__device__ __forceinline__ void k1_item(const float4 vr, const float4 vg, const float4 vb, const K1Tables& t,
                                        unsigned char* s_cnt, uint32_t tid4, uint32_t& wl, uint32_t& wa, uint32_t& wb)
{
    const float pr[4] = {vr.x, vr.y, vr.z, vr.w};
    const float pg[4] = {vg.x, vg.y, vg.z, vg.w};
    const float pb[4] = {vb.x, vb.y, vb.z, vb.w};
    uint32_t m0 = __vimax3_u32(__float_as_uint(pr[0]), __float_as_uint(pr[1]), __float_as_uint(pr[2]));
    uint32_t m1 = __vimax3_u32(__float_as_uint(pr[3]), __float_as_uint(pg[0]), __float_as_uint(pg[1]));
    uint32_t m2 = __vimax3_u32(__float_as_uint(pg[2]), __float_as_uint(pg[3]), __float_as_uint(pb[0]));
    uint32_t m3 = __vimax3_u32(__float_as_uint(pb[1]), __float_as_uint(pb[2]), __float_as_uint(pb[3]));
    m0 = __vimax3_u32(m0, m1, m2);
    m0 = max(m0, m3);
    float R[4], G[4], B[4];
    if (m0 <= 0x3F800000u) {   // every value in [+0, 1]: as unsigned integers, positive floats order like their values
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            R[k] = lds_f32(__float_as_uint(__fadd_rz(__fmul_rn(pr[k], 255.0f), 8388608.0f)) * 4u + t.gam_q);
            G[k] = lds_f32(__float_as_uint(__fadd_rz(__fmul_rn(pg[k], 255.0f), 8388608.0f)) * 4u + t.gam_q);
            B[k] = lds_f32(__float_as_uint(__fadd_rz(__fmul_rn(pb[k], 255.0f), 8388608.0f)) * 4u + t.gam_q);
        }
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            R[k] = lds_f32(uint32_t(quantize_u8(pr[k])) * 4u + t.gam);
            G[k] = lds_f32(uint32_t(quantize_u8(pg[k])) * 4u + t.gam);
            B[k] = lds_f32(uint32_t(quantize_u8(pb[k])) * 4u + t.gam);
        }
    }
    k1_core(R, G, B, t, s_cnt, tid4, wl, wa, wb);
}

// 12 packed bytes (4 px x RGB, HWC order: R0 G0 B0 R1 | G1 B1 R2 G2 | B2 R3 G3 B3) -> three Lab words + four counter increments
__device__ __forceinline__ void k1_item_u8(uint32_t w0, uint32_t w1, uint32_t w2, const K1Tables& t, unsigned char* s_cnt,
                                           uint32_t tid4, uint32_t& wl, uint32_t& wa, uint32_t& wb)
{
    // byte k of a word, times four, is ((w >> (8k - 2)) & 0x3FC): the gamma table is indexed by the byte itself
    auto gam = [&](uint32_t w, int k) {
        const uint32_t off = k == 0 ? (w << 2) & 0x3FCu : (w >> (8 * k - 2)) & 0x3FCu;
        return lds_f32(off + t.gam);
    };
    const float R[4] = {gam(w0, 0), gam(w0, 3), gam(w1, 2), gam(w2, 1)};
    const float G[4] = {gam(w0, 1), gam(w1, 0), gam(w1, 3), gam(w2, 2)};
    const float B[4] = {gam(w0, 2), gam(w1, 1), gam(w2, 0), gam(w2, 3)};
    k1_core(R, G, B, t, s_cnt, tid4, wl, wa, wb);
}

// gamma-table values of 4 pixels (exact small integers in fp32) -> three Lab words + four counter increments
__device__ __forceinline__ void k1_core(const float (&R)[4], const float (&G)[4], const float (&B)[4], const K1Tables& t,
                                        unsigned char* s_cnt, uint32_t tid4, uint32_t& wl, uint32_t& wa, uint32_t& wb)
{
    int vL[4], vA[4], vB[4], fY[4];
    // Y first: L only needs fY, and the four counter updates then overlap the X/Z arithmetic instead of trailing it
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        // S = c0 R + c1 G + c2 B + 2048 is an exact integer < 2^24; RZ(S / 4096 + 2^23) carries floor(S / 4096)
        const float sy = __fmaf_rn(B[k], 296.0f, __fmaf_rn(G[k], 2929.0f, __fmaf_rn(R[k], 871.0f, 2048.0f)));
        fY[k] = int(lds_u16(__float_as_uint(__fmaf_rz(sy, 0.000244140625f, 8388608.0f)) * 2u + t.cbr_q));
        // twice the Appendix A.1 expressions: the u8 result is byte 2 (L 0..255, a 42..226, b 20..223, never negative)
        vL[k] = fY[k] * 592 - 2641100;                 // 2 * (296 fY - 1336934 + 16384)
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        // L sits in byte 2 of vL: one PRMT copies it into bytes 0 and 1 (= L * 257), which masked with 0xFC00 is the row
        // of its counter word.  The four byte counters of a word belong to ONE thread and never exceed 255 between
        // flushes, so adding 1 << 8 (L & 3) to the word with a shared-memory reduction cannot carry: one LSU operation
        // instead of a dependent byte load / add / store (bits 2..9 of the offset are the thread's column: no conflicts)
        const uint32_t a = uint32_t(__cvta_generic_to_shared(s_cnt)) + ((__byte_perm(uint32_t(vL[k]), 0u, 0x4422) & 0xFC00u) | tid4);
        const uint32_t inc = 1u << ((uint32_t(vL[k]) >> 13) & 24u);
        asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(inc) : "memory");
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float sx = __fmaf_rn(B[k], 778.0f, __fmaf_rn(G[k], 1541.0f, __fmaf_rn(R[k], 1777.0f, 2048.0f)));
        const float sz = __fmaf_rn(B[k], 3575.0f, __fmaf_rn(G[k], 448.0f, __fmaf_rn(R[k], 73.0f, 2048.0f)));
        const int fX = int(lds_u16(__float_as_uint(__fmaf_rz(sx, 0.000244140625f, 8388608.0f)) * 2u + t.cbr_q));
        const int fZ = int(lds_u16(__float_as_uint(__fmaf_rz(sz, 0.000244140625f, 8388608.0f)) * 2u + t.cbr_q));
        vA[k] = (fX - fY[k]) * 1000 + 8421376;         // 2 * (500 (fX - fY) + 128 * 32768 + 16384)
        vB[k] = (fY[k] - fZ) * 400 + 8421376;
    }
    wl = __byte_perm(__byte_perm(uint32_t(vL[0]), uint32_t(vL[1]), 0x0062), __byte_perm(uint32_t(vL[2]), uint32_t(vL[3]), 0x0062), 0x5410);
    wa = __byte_perm(__byte_perm(uint32_t(vA[0]), uint32_t(vA[1]), 0x0062), __byte_perm(uint32_t(vA[2]), uint32_t(vA[3]), 0x0062), 0x5410);
    wb = __byte_perm(__byte_perm(uint32_t(vB[0]), uint32_t(vB[1]), 0x0062), __byte_perm(uint32_t(vB[2]), uint32_t(vB[3]), 0x0062), 0x5410);
}

// kFused: the CLAHE input is the Retinex recombination of the CNN outputs (models/model.py:405-413,442 followed by
// adaptive_params.py:195): enhanced = R*e + (1-R)*e^2 with R = x / (illu + eps), evaluated in registers with exactly the
// arithmetic of k_recombine_vec (upr_maps.cuh: IEEE division, separately rounded products, the roundings of the map dtypes) --
// the 12 B/px `enhanced` frame is never written nor re-read (x 12 + illu 4 + e 12 B/px are read instead, less for fp16 / bf16
// maps).  The pointers have the kernel's map types TI (illu) and TE (e).
struct RetinexIn {
    const void* illu;    // [n][1][h][w]
    const void* e;       // [n][3][h][w]
    float eps;
};

// ---------------------------------------------------------------------------------------------
// K1 fast path kernel: COLUMN-OWNER threads.  One CTA per (frame, tile, row strip).  The first
// nact = (256 / (tw/4)) * (tw/4) threads of the CTA own one 4-pixel column each and walk down the strip
// rpi = 256 / (tw/4) rows at a time (1080p and 4K: 240 threads, 4 resp. 2 rows): ONE 32-bit group offset advances by a
// constant, every address is one IMAD.WIDE.U32 against a per-thread base, the L2 prefetch target is the same offset plus a
// constant.  (Spare threads idle in the main loop and own a histogram bin in the epilogue; tiles wider than 1024 px are
// walked in passes of 256 columns.)  An item-linear predecessor spent 57 of its 224 instructions per 4-pixel item on
// row / column wrap bookkeeping for its three pointer sets.  The kernel is bound by its memory streams and the L1/shared
// data pipe, not by issue (profiles/r3_clahe.md).
//   kU8In : the frame is packed u8 RGB (HWC, upr_clahe_lab_u8): a 4-pixel group is 12 contiguous bytes, three 32-bit
//           loads; the bytes index the gamma table directly (no quantisation).
//   kFused: the CLAHE input is the Retinex recombination of the CNN outputs (models/model.py:405-413,442 followed by
//           adaptive_params.py:195), evaluated in registers (recombine1) from x, illu and e: 28 B/px read (f32 maps)
//           instead of a 12 B/px `enhanced` frame written by one kernel and re-read by this one.  One raw register set
//           requested one iteration ahead (f32 maps: 7 float4; fp16 / bf16 e: 8 bytes per 4 pixels and channel, kept packed
//           until use); two CTAs per SM (128 registers) instead of three.  TI / TE / kAutocast: the maps' dtypes and
//           autocast semantics of e**2 (upr_maps.cuh).
// ---------------------------------------------------------------------------------------------
template <bool kU8In, bool kFused, typename TI = float, typename TE = float, bool kAutocast = false>
__global__ void __launch_bounds__(kK1Threads, kFused ? 2 : 3)
k_hist_lab_vec3(const void* __restrict__ in, uint8_t* __restrict__ lab, int32_t* __restrict__ hist_g,
                uint8_t* __restrict__ lut_g, unsigned* __restrict__ tickets, const ClaheGeom g, const RetinexIn rx)
{
    static_assert(!(kU8In && kFused), "the fused Retinex prologue reads f32 planes");
    extern __shared__ __align__(16) unsigned char smem[];
    unsigned char* s_cnt = smem;                                                   // [64 bin groups][256 threads][4 bins] u8
    float* s_gammaf = reinterpret_cast<float*>(smem + 256 * kK1Threads);           // 256 x f32
    uint16_t* s_cbrt = reinterpret_cast<uint16_t*>(s_gammaf + UPR_TAB_GAMMA_LEN);  // 2048 x u16
    __shared__ int s_tmp[8];
    __shared__ int s_flag;

    const int tid = threadIdx.x;
    const int strip = blockIdx.x % g.nstrips;
    const int tile = blockIdx.x / g.nstrips;
    const int ty = tile / g.tiles_x, tx = tile - ty * g.tiles_x;
    const int f = blockIdx.y;
    const int ntiles = g.tiles_x * g.tiles_y;

    {
        uint4* z = reinterpret_cast<uint4*>(s_cnt);
#pragma unroll
        for (int i = 0; i < 256 * kK1Threads / 16 / kK1Threads; ++i) z[tid + i * kK1Threads] = make_uint4(0, 0, 0, 0);
        s_gammaf[tid] = float(d_gamma[tid]);
        reinterpret_cast<uint4*>(s_cbrt)[tid] = reinterpret_cast<const uint4*>(d_cbrt)[tid];  // 256 x 16 B = 4 KB
    }
    __syncthreads();

    const uint32_t zero = blockIdx.z;  // always 0
    K1Tables t;
    t.gam = uint32_t(__cvta_generic_to_shared(s_gammaf));
    t.gam_q = t.gam + g.gam_bias;
    t.cbr_q = opaque(uint32_t(__cvta_generic_to_shared(s_cbrt)) - 2u * 0x4B000000u);
    t.four = opaque(4u + zero);
    t.sixteen = opaque(16u + zero);

    const int tw4 = g.tw >> 2;
    const int cpp = min(tw4, kK1Threads);          // columns per pass (one pass unless the tile is wider than 1024 px)
    const int rpi = kK1Threads / cpp;              // rows per iteration
    const int lr = tid / cpp, lc0 = tid - lr * cpp;
    const int row0 = ty * g.th + strip * g.strip_rows;
    const int strip_end = min(row0 + g.strip_rows, (ty + 1) * g.th);
    const uint32_t w4 = uint32_t(g.w) >> 2;
    const uint32_t plane4 = (uint32_t(g.h) * uint32_t(g.w)) >> 2;      // fast path: 3 * plane < 2^32
    const uint32_t step = uint32_t(rpi) * w4;
    // L2 prefetch distance in iterations (of rpi rows).  Swept on 64 x 1080p (rpi = 4): 1 -> 0.473 ms, 2 and 3 -> 0.381 ms,
    // 4 -> 0.385, 6 -> 0.394, 8 -> 0.402, 14 -> 0.430, 20 -> 0.459; 16 x 4K (rpi = 2) is flat between 3 and 6
    constexpr int kPf = 3;
    const uint32_t pfo = uint32_t(kPf) * step;
    const uint32_t tid4 = uint32_t(tid) * 4u;

#pragma unroll 1
    for (int xc = 0; xc < tw4; xc += cpp) {
    const int lc = xc + lc0;
    const int row1 = (lr < rpi && lc < tw4) ? strip_end : 0;   // spare threads: empty range
    // per-THREAD plane bases (frame, tile column, this thread's 4-pixel column): a base that lives in vector registers
    // lets ptxas address base[o] with one IMAD.WIDE.U32 (block-uniform bases end up in uniform registers and cost a
    // shift, a multiply-high and two 64-bit adds per access).  Row offsets count 4-pixel groups: a float4 of the input
    // and a u32 word of the Lab planes share the same index.
    // (opaque_ptr: otherwise the front end re-associates base + (K + o) back onto the kernel parameter)
    const uint32_t col = uint32_t(tx * tw4 + lc);
    const float4* inR = opaque_ptr(reinterpret_cast<const float4*>(in) + (size_t(f) * 3 * plane4 + col));
    const float4* inG = opaque_ptr(inR + plane4);
    const float4* inB = opaque_ptr(inG + plane4);
    struct Px4 { uint32_t w[3]; };   // one 4-pixel group of a packed u8 frame
    const Px4* in8 = opaque_ptr(reinterpret_cast<const Px4*>(in) + (size_t(f) * plane4 + col));
    uint32_t* labL = opaque_ptr(reinterpret_cast<uint32_t*>(lab) + (size_t(f) * 3 * plane4 + col));
    uint32_t* labA = opaque_ptr(labL + plane4);
    uint32_t* labB = opaque_ptr(labA + plane4);

    auto store = [&](uint32_t o, uint32_t wl, uint32_t wa, uint32_t wb) {
        st_global_u32(labL + o, wl);
        st_global_u32(labA + o, wa);
        st_global_u32(labB + o, wb);
    };

    int row = row0 + lr;
    uint32_t o = uint32_t(row) * w4;
    const int row_ld = row1 - rpi;                  // row < row_ld: there is a next iteration to load
    const int row_pf = row1 - kPf * rpi;            // row < row_pf: there is an iteration kPf ahead to prefetch

    if constexpr (kFused) {
        using RawE = typename MapIO<TE>::Raw4;
        using RawI = typename MapIO<TI>::Raw4;
        const RawE* eR = opaque_ptr(reinterpret_cast<const RawE*>(rx.e) + (size_t(f) * 3 * plane4 + col));
        const RawE* eG = opaque_ptr(eR + plane4);
        const RawE* eB = opaque_ptr(eG + plane4);
        const RawI* ilp = opaque_ptr(reinterpret_cast<const RawI*>(rx.illu) + (size_t(f) * plane4 + col));
        float4 X0, X1, X2;
        RawE E0, E1, E2;
        RawI IL;
        auto load7 = [&](uint32_t oo) {
            X0 = ld_nc_f4(inR + oo); X1 = ld_nc_f4(inG + oo); X2 = ld_nc_f4(inB + oo);
            E0 = MapIO<TE>::ld4nc(eR + oo); E1 = MapIO<TE>::ld4nc(eG + oo); E2 = MapIO<TE>::ld4nc(eB + oo);
            IL = MapIO<TI>::ld4nc(ilp + oo);
        };
        auto prefetch7 = [&](uint32_t oo) {
            prefetch_l2(inR + oo); prefetch_l2(inG + oo); prefetch_l2(inB + oo);
            prefetch_l2(eR + oo); prefetch_l2(eG + oo); prefetch_l2(eB + oo);
            prefetch_l2(ilp + oo);
        };
        auto recombine4 = [&](const float4 xv, const RawE raw, const float d[4]) {
            const float4 ev = MapIO<TE>::wide4(raw);
            float4 r;
            float refl;
            recombine1<TE, kAutocast>(xv.x, d[0], ev.x, refl, r.x);
            recombine1<TE, kAutocast>(xv.y, d[1], ev.y, refl, r.y);
            recombine1<TE, kAutocast>(xv.z, d[2], ev.z, refl, r.z);
            recombine1<TE, kAutocast>(xv.w, d[3], ev.w, refl, r.w);
            return r;
        };
        if (row < row1) {
            load7(o);
#pragma unroll 1
            for (int k = 1; k < kPf; ++k)
                if (row + k * rpi < row1) prefetch7(o + uint32_t(k) * step);
        }
        while (row < row1) {
            const float4 il = MapIO<TI>::wide4(IL);
            const float d[4] = {illu_eps<TI>(il.x, rx.eps), illu_eps<TI>(il.y, rx.eps), illu_eps<TI>(il.z, rx.eps),
                                illu_eps<TI>(il.w, rx.eps)};
            const float4 er = recombine4(X0, E0, d), eg = recombine4(X1, E1, d), eb = recombine4(X2, E2, d);
            if (row < row_ld) load7(o + step);
            if (row < row_pf) prefetch7(o + pfo);
            uint32_t wl, wa, wb;
            k1_item(er, eg, eb, t, s_cnt, tid4, wl, wa, wb);
            store(o, wl, wa, wb);
            row += rpi;
            o += step;
        }
    } else {
        // (u8 frames: the three words of a group travel in the .x lanes of the three float4 registers)
        auto load = [&](uint32_t oo, float4& r, float4& gch, float4& b) {
            if constexpr (kU8In) {
                r.x = __uint_as_float(ld_nc_u32p(&in8[oo].w[0]));
                gch.x = __uint_as_float(ld_nc_u32p(&in8[oo].w[1]));
                b.x = __uint_as_float(ld_nc_u32p(&in8[oo].w[2]));
            } else {
                r = ld_nc_f4(inR + oo);
                gch = ld_nc_f4(inG + oo);
                b = ld_nc_f4(inB + oo);
            }
        };
        auto prefetch = [&](uint32_t oo) {
            if constexpr (kU8In) {
                prefetch_l2(in8 + oo);
            } else {
                prefetch_l2(inR + oo);
                prefetch_l2(inG + oo);
                prefetch_l2(inB + oo);
            }
        };
        auto item = [&](const float4& r, const float4& gch, const float4& b, uint32_t& wl, uint32_t& wa, uint32_t& wb) {
            if constexpr (kU8In) k1_item_u8(__float_as_uint(r.x), __float_as_uint(gch.x), __float_as_uint(b.x), t, s_cnt, tid4, wl, wa, wb);
            else k1_item(r, gch, b, t, s_cnt, tid4, wl, wa, wb);
        };
        // two register sets: the twelve floats of iteration i+1 are in flight while iteration i is converted
        float4 ar, ag, ab, br, bg, bb;
        if (row < row1) {
            load(o, ar, ag, ab);
#pragma unroll 1
            for (int k = 1; k < kPf; ++k)
                if (row + k * rpi < row1) prefetch(o + uint32_t(k) * step);
        }
        while (row < row1) {
            uint32_t wl, wa, wb;
            if (row < row_ld) load(o + step, br, bg, bb);
            if (row < row_pf) prefetch(o + pfo);
            item(ar, ag, ab, wl, wa, wb);
            store(o, wl, wa, wb);
            row += rpi;
            o += step;
            if (row >= row1) break;
            if (row < row_ld) load(o + step, ar, ag, ab);
            if (row < row_pf) prefetch(o + pfo);
            item(br, bg, bb, wl, wa, wb);
            store(o, wl, wa, wb);
            row += rpi;
            o += step;
        }
    }
    }
    __syncthreads();

    // thread `tid` sums bin `tid`: byte (tid&3) of the 256 words of row (tid>>2).  The four threads of a
    // row read the same 16-byte chunks (broadcast); chunk order is rotated by the row so that the eight
    // rows of a warp hit disjoint banks.
    unsigned total_u = 0;
    {
        const uint4* rowp = reinterpret_cast<const uint4*>(s_cnt + (tid >> 2) * (kK1Threads * 4));
        const unsigned sel = 1u << (8 * (tid & 3));
#pragma unroll 8
        for (int k = 0; k < kK1Threads / 4; ++k) {
            const uint4 v = rowp[(k + (tid >> 2)) & (kK1Threads / 4 - 1)];
            total_u = __dp4a(v.x, sel, total_u);
            total_u = __dp4a(v.y, sel, total_u);
            total_u = __dp4a(v.z, sel, total_u);
            total_u = __dp4a(v.w, sel, total_u);
        }
    }
    int total = int(total_u);
    const size_t t_idx = size_t(f) * ntiles + tile;
    if (!publish_hist(total, hist_g + t_idx * 256, tickets + t_idx, g.nstrips, &s_flag)) return;
    tile_lut_256(total, g.clip, g.lut_scale, lut_g + t_idx * 256, s_tmp);
}

// ---------------------------------------------------------------------------------------------
// K1 generic path: any size (including OpenCV's reflect-101 padding quirk, Appendix A.3 step 1).
// One CTA per (frame, tile); per-warp shared histograms with atomics.  Correctness path for
// ragged shapes -- the named workloads all take the vector path.
//   kFused: as in k_hist_lab_vec3, the input is the Retinex recombination of x, illu (TI) and e (TE), evaluated per
//           (reflected) pixel with recombine1; each map value is widened where it is loaded.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect101(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * (len - 1) - p;
    return p;
}

template <bool kU8In, bool kFused, typename TI = float, typename TE = float, bool kAutocast = false>
__global__ void __launch_bounds__(256)
k_hist_lab_generic(const void* __restrict__ in, uint8_t* __restrict__ lab, int32_t* __restrict__ hist_g,
                   uint8_t* __restrict__ lut_g, const ClaheGeom g, const RetinexIn rx)
{
    static_assert(!(kU8In && kFused), "the fused Retinex prologue reads f32 planes");
    __shared__ int s_hist[8][256];
    __shared__ uint16_t s_gamma[UPR_TAB_GAMMA_LEN];
    __shared__ uint16_t s_cbrt[UPR_TAB_CBRT_LEN];
    __shared__ int s_tmp[8];

    const int tid = threadIdx.x, wid = tid >> 5;
    const int tile = blockIdx.x;
    const int ty = tile / g.tiles_x, tx = tile - ty * g.tiles_x;
    const int f = blockIdx.y;
    const int ntiles = g.tiles_x * g.tiles_y;
    for (int i = tid; i < 8 * 256; i += 256) (&s_hist[0][0])[i] = 0;
    s_gamma[tid] = d_gamma[tid];
    for (int i = tid; i < UPR_TAB_CBRT_LEN; i += 256) s_cbrt[i] = d_cbrt[i];
    __syncthreads();

    const size_t plane = size_t(g.h) * g.w;
    const float* inR = reinterpret_cast<const float*>(in) + size_t(f) * 3 * plane;
    const uint8_t* in8 = reinterpret_cast<const uint8_t*>(in) + size_t(f) * 3 * plane;   // kU8In: packed RGB (HWC)
    uint8_t* labL = lab + size_t(f) * 3 * plane;
    const int area = g.tw * g.th;
    const uint64_t pol_stream = policy_evict_first();
    for (int i = tid; i < area; i += 256) {
        const int py = ty * g.th + i / g.tw, px = tx * g.tw + i % g.tw;
        const bool inside = py < g.h && px < g.w;
        const size_t off = size_t(reflect101(py, g.h)) * g.w + reflect101(px, g.w);
        int qr, qg, qb;
        if constexpr (kU8In) {
            qr = in8[3 * off + 0]; qg = in8[3 * off + 1]; qb = in8[3 * off + 2];
        } else if constexpr (kFused) {
            const TE* eR = static_cast<const TE*>(rx.e) + size_t(f) * 3 * plane;
            const float d = illu_eps<TI>(MapIO<TI>::ld1(static_cast<const TI*>(rx.illu) + size_t(f) * plane + off, pol_stream), rx.eps);
            float refl, o[3];
#pragma unroll
            for (int c = 0; c < 3; ++c)
                recombine1<TE, kAutocast>(ld_stream_f1(inR + c * plane + off, pol_stream), d, MapIO<TE>::ld1(eR + c * plane + off, pol_stream),
                                          refl, o[c]);
            qr = quantize_u8(o[0]); qg = quantize_u8(o[1]); qb = quantize_u8(o[2]);
        } else {
            qr = quantize_u8(ld_stream_f1(inR + off, pol_stream));
            qg = quantize_u8(ld_stream_f1(inR + plane + off, pol_stream));
            qb = quantize_u8(ld_stream_f1(inR + 2 * plane + off, pol_stream));
        }
        int L;
        if (inside) {
            int a, b;
            rgb_to_lab(qr, qg, qb, s_gamma, s_cbrt, L, a, b);
            labL[off] = uint8_t(L);
            labL[plane + off] = uint8_t(a);
            labL[2 * plane + off] = uint8_t(b);
        } else {
            L = rgb_to_l_only(qr, qg, qb, s_gamma, s_cbrt);
        }
        atomicAdd(&s_hist[wid][L], 1);
    }
    __syncthreads();
    int total = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) total += s_hist[k][tid];
    const size_t t_idx = size_t(f) * ntiles + tile;
    hist_g[t_idx * 256 + tid] = total;
    tile_lut_256(total, g.clip, g.lut_scale, lut_g + t_idx * 256, s_tmp);
}

// ---------------------------------------------------------------------------------------------
// K3 fast path.  Experiments on an earlier one-CTA-per-item version (profiles/r2_*): with loads AND stores suppressed the
// kernel still took 0.40 of 0.44 ms -- it is bound by instruction issue (94 executed instructions per pixel incl.
// prologues and idle lanes), not by HBM or by shared-memory bank conflicts (constant frames are as slow as noise).
// Hence a short instruction stream:
//   * abToXZ: the cubic branch is 4 instructions; the linear branch (i <= 3390: C truncating division, 7 instructions
//     plus a select) becomes a PREDICATED 16-bit table load (23 KB table; only dark pixels take it, so the gather is
//     sparse);
//   * {ify - 4194, y} of a grey level come from one 64-bit shared load, nothing to unpack;
//   * the CTA has a multiple of the cell width in threads (240-px cell = 60 four-pixel columns -> 480 threads = 8 full
//     rows): no idle lanes (first generations: 16 of 256);
//   * persistent CTAs (2 per SM) pull (frame, cell, strip) items from an atomic counter: the 41 KB of tables are staged
//     once per CTA instead of once per item, no tail wave; the quad table of the next item is built while the current
//     one is mapped (one barrier per item).
// Arithmetic: Appendix A.2 / A.3 (the generic kernel k_map_generic states it in plain C).
// ---------------------------------------------------------------------------------------------
constexpr int kK5MaxThreads = 512;
constexpr int kXzLinMin = -8145;
constexpr int kXzLinBytes = (UPR_TAB_XZLIN_LEN * 2 + 15) / 16 * 16;

struct Map5Tables {
    uint32_t four;      // 4, opaque to ptxas
    uint32_t quad;      // shared address of the current quad table (u32[256])
    uint32_t ay_lp;     // &s_ay[0] - 0x4B400000*8: address of {A, y}[L'] straight from the magic-add bits
    uint32_t outf;      // shared address of float[4096]
    uint32_t lin;       // &s_lin[0] - 2*kXzLinMin
};

__device__ __forceinline__ int ab_to_xz5(int i, uint32_t lin)
{
    int x = (((i * i) >> 14) * i) >> 14;
    asm("{\n\t.reg .pred p;\n\tsetp.le.s32 p, %1, 3390;\n\t@p ld.shared.s16 %0, [%2];\n\t}" : "+r"(x) : "r"(i), "r"(uint32_t(i) * 2u + lin));
    return x;
}

// kU8Out: the three results are the u8 channel values (integers in the bit patterns of r, g, b) instead of value / 255
template <uint32_t kAyStride, bool kU8Out>
__device__ __forceinline__ void map_pixel5(uint32_t Lv, int av, int bv, float xa, float xa1, float ya, float ya1,
                                           const Map5Tables& t, float& r, float& g, float& b)
{
    const uint32_t q = lds_u32(Lv * t.four + t.quad);
    const float l11 = float(q & 0xffu), l12 = float((q >> 8) & 0xffu), l21 = float((q >> 16) & 0xffu), l22 = float(q >> 24);
    const float top = __fadd_rn(__fmul_rn(l11, xa1), __fmul_rn(l12, xa));
    const float bot = __fadd_rn(__fmul_rn(l21, xa1), __fmul_rn(l22, xa));
    const float res = __fadd_rn(__fmul_rn(top, ya1), __fmul_rn(bot, ya));
    // rint via 1.5*2^23 (round-half-even == cvRound); 0 <= res < 255.5, so the sum's bits are 0x4B400000 + L'
    int A, y;
    asm("ld.shared.v2.s32 {%0,%1}, [%2];" : "=r"(A), "=r"(y) : "r"(__float_as_uint(__fadd_rn(res, 12582912.0f)) * kAyStride + t.ay_lp));
    // ix = ify + adiv(a);  iz = ify - bdiv(b) = A + 14678 - ((b*41943+16) >> 9)  with  -(u >> 9) == (511 - u) >> 9
    const int x = ab_to_xz5(A + ((av * 268435 + 128) >> 13), t.lin);
    const int z = ab_to_xz5(A + ((bv * -41943 + (495 + 14678 * 512)) >> 9), t.lin);
    const int ro = __vimin_s32_relu((12615 * x - 6296 * y - 2223 * z + 8192) >> 14, 4095);
    const int go = __vimin_s32_relu((-3773 * x + 7684 * y + 185 * z + 8192) >> 14, 4095);
    const int bo = __vimin_s32_relu((217 * x - 836 * y + 4715 * z + 8192) >> 14, 4095);
    if constexpr (kU8Out) {
        uint32_t ur, ug, ub;
        asm("ld.shared.u8 %0, [%1];" : "=r"(ur) : "r"(uint32_t(ro) + t.outf));
        asm("ld.shared.u8 %0, [%1];" : "=r"(ug) : "r"(uint32_t(go) + t.outf));
        asm("ld.shared.u8 %0, [%1];" : "=r"(ub) : "r"(uint32_t(bo) + t.outf));
        r = __uint_as_float(ur); g = __uint_as_float(ug); b = __uint_as_float(ub);
    } else {
        r = lds_f32(uint32_t(ro) * t.four + t.outf);
        g = lds_f32(uint32_t(go) * t.four + t.outf);
        b = lds_f32(uint32_t(bo) * t.four + t.outf);
    }
}

// kAyRep: the {A, y} table is replicated 16 times ([grey level][lane & 15], 32 KB): its 64-bit gather is served half a
// warp at a time, so with one copy per lane of a half-warp it is conflict-free (measured 4.4 wavefronts per gather with
// the plain table).
// kU8Out: the result is a packed u8 RGB frame (HWC; upr_clahe_lab_u8 / upr_clahe_lab_f32_u8): u8 inverse-gamma table, 12 bytes per
// 4-pixel group in three 32-bit stores.
template <bool kAyRep, bool kU8Out>
__global__ void __launch_bounds__(kK5MaxThreads, 2)
k_map_vec5(const uint8_t* __restrict__ lab, const uint8_t* __restrict__ lut_g, void* __restrict__ out, const MapGeom g,
           unsigned* __restrict__ work, int nitems)
{
    extern __shared__ __align__(16) unsigned char smem5[];
    int16_t* s_lin = reinterpret_cast<int16_t*>(smem5);
    float* s_outf = reinterpret_cast<float*>(smem5 + kXzLinBytes);
    int* s_ay = reinterpret_cast<int*>(s_outf + 4096);             // {A, y}[256]
    uint32_t* s_quad = reinterpret_cast<uint32_t*>(s_ay + 512 * (kAyRep ? 16 : 1));    // [2][256]
    __shared__ int s_nxt[2];

    const int tid = threadIdx.x, nthr = blockDim.x;
    auto build_quad = [&](int item, uint32_t* dst) {   // tid < 256
        int f, cell, strip_unused;
        map_item(g, item, f, cell, strip_unused);
        const int cy = cell / (g.tiles_x + 1), cx = cell - cy * (g.tiles_x + 1);
        const int ty1 = max(cy - 1, 0), ty2 = min(cy, g.tiles_y - 1);
        const int tx1 = max(cx - 1, 0), tx2 = min(cx, g.tiles_x - 1);
        const uint8_t* lf = lut_g + size_t(f) * g.tiles_x * g.tiles_y * 256 + tid;
        dst[tid] = uint32_t(lf[(ty1 * g.tiles_x + tx1) * 256]) | (uint32_t(lf[(ty1 * g.tiles_x + tx2) * 256]) << 8) |
                   (uint32_t(lf[(ty2 * g.tiles_x + tx1) * 256]) << 16) | (uint32_t(lf[(ty2 * g.tiles_x + tx2) * 256]) << 24);
    };

    int cur = blockIdx.x;
    {
        for (int i = tid; i < kXzLinBytes / 16; i += nthr) reinterpret_cast<uint4*>(s_lin)[i] = reinterpret_cast<const uint4*>(d_xzlin)[i];
        if constexpr (kU8Out) {   // u8 results: the 4 KB inverse-gamma table itself (first quarter of the same slot)
            for (int i = tid; i < 256; i += nthr) reinterpret_cast<uint4*>(s_outf)[i] = reinterpret_cast<const uint4*>(d_invgamma)[i];
        } else {
            for (int i = tid; i < 1024; i += nthr) reinterpret_cast<uint4*>(s_outf)[i] = reinterpret_cast<const uint4*>(d_outf_bits)[i];
        }
        if constexpr (kAyRep) {
            for (int i = tid; i < 256 * 16; i += nthr) {
                const uint32_t yf = d_labyf[i >> 4];
                reinterpret_cast<int2*>(s_ay)[i] = make_int2(int(yf & 0xffffu) - 4194, int(yf >> 16));
            }
        }
        if (tid < 256) {
            if constexpr (!kAyRep) {
                const uint32_t yf = d_labyf[tid];
                s_ay[tid * 2 + 0] = int(yf & 0xffffu) - 4194;
                s_ay[tid * 2 + 1] = int(yf >> 16);
            }
            if (cur < nitems) build_quad(cur, s_quad);
        }
        if (tid == 0) s_nxt[0] = int(gridDim.x + atomicAdd(work, 1u));
    }
    __syncthreads();

    Map5Tables t;
    const uint32_t zero = blockIdx.z;  // always 0
    t.four = opaque(4u + zero);
    constexpr uint32_t kAyStride = kAyRep ? 128u : 8u;
    t.ay_lp = kAyRep ? uint32_t(__cvta_generic_to_shared(s_ay)) + uint32_t(tid & 15) * 8u + g.ay_bias
                     : opaque(uint32_t(__cvta_generic_to_shared(s_ay)) - 0x4B400000u * 8u);
    t.outf = opaque(uint32_t(__cvta_generic_to_shared(s_outf)));
    t.lin = opaque(uint32_t(__cvta_generic_to_shared(s_lin)) - 2u * uint32_t(kXzLinMin));
    const uint32_t sixteen = opaque(16u + zero);
    const uint32_t quad0 = uint32_t(__cvta_generic_to_shared(s_quad));

    const uint32_t plane4 = (uint32_t(g.h) * uint32_t(g.w)) >> 2;
    const uint32_t w4 = uint32_t(g.w) >> 2;

    for (int buf = 0; cur < nitems; buf ^= 1) {
        const int nxt = s_nxt[buf];
        if (nxt < nitems && tid < 256) build_quad(nxt, s_quad + (buf ^ 1) * 256);
        if (tid == 0) s_nxt[buf ^ 1] = int(gridDim.x + atomicAdd(work, 1u));
        t.quad = quad0 + uint32_t(buf) * 1024u;

        int f, cell, strip;
        map_item(g, cur, f, cell, strip);
        const int cy = cell / (g.tiles_x + 1), cx = cell - cy * (g.tiles_x + 1);
        const int x0 = g.bx[cx], x1 = g.bx[cx + 1];
        const int rows_cell = g.by[cy + 1] - g.by[cy];
        const int srows = (rows_cell + g.nstrips - 1) / g.nstrips;
        const int y0 = g.by[cy] + strip * srows;
        const int y1 = min(y0 + srows, g.by[cy + 1]);

        const uint32_t* labL = reinterpret_cast<const uint32_t*>(lab) + size_t(f) * 3 * plane4;
        // bytes per 4-pixel group of the result: 16 (one float4 per plane) or 12 (packed u8 RGB)
        constexpr uint32_t kOB = kU8Out ? 12u : 16u;
        char* outF = reinterpret_cast<char*>(out) + size_t(f) * (kU8Out ? 1 : 3) * plane4 * kOB;
        const float txbase = float(cx - 1), tybase = float(cy - 1);
        const int cw4 = (x1 - x0) >> 2;

        for (int xc = 0; xc < cw4; xc += nthr) {
            const int cwc = min(nthr, cw4 - xc);
            const int rpi = nthr / cwc;  // rows per iteration
            const int lr = tid / cwc, lc = tid - lr * cwc;
            if (lr >= rpi) continue;
            const int x = x0 + (xc + lc) * 4;
            float xa[4], xa1[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float txf = __fadd_rn(__fmul_rn(float(x + k), g.inv_tw), -0.5f);
                xa[k] = __fsub_rn(txf, txbase);
                xa1[k] = __fsub_rn(1.0f, xa[k]);
            }
            // per-thread 64-bit row pointers, advanced by a constant byte stride (2 instructions per plane and row)
            const char* pl = reinterpret_cast<const char*>(labL + (uint32_t(y0 + lr) * w4 + (uint32_t(x) >> 2)));
            char* po = outF + size_t(uint32_t(y0 + lr) * w4 + (uint32_t(x) >> 2)) * kOB;
            const uint32_t step4 = uint32_t(rpi) * w4;   // row stride of this thread in 4-pixel groups

            auto load3 = [&](const char* p, uint32_t& l, uint32_t& a, uint32_t& b) {
                l = __ldg(reinterpret_cast<const uint32_t*>(p));
                a = __ldg(reinterpret_cast<const uint32_t*>(wide_imm<4>(p, plane4)));
                b = __ldg(reinterpret_cast<const uint32_t*>(wide_imm<8>(p, plane4)));
            };
            auto map_row = [&](int y, char* p, uint32_t wl, uint32_t wa, uint32_t wb) {
                const float tyf = __fadd_rn(__fmul_rn(float(y), g.inv_th), -0.5f);
                const float ya = __fsub_rn(tyf, tybase);
                const float ya1 = __fsub_rn(1.0f, ya);
                float o[3][4];
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    map_pixel5<kAyStride, kU8Out>(__byte_perm(wl, 0u, 0x4440u | uint32_t(k)), int(__byte_perm(wa, 0u, 0x4440u | uint32_t(k))),
                               int(__byte_perm(wb, 0u, 0x4440u | uint32_t(k))), xa[k], xa1[k], ya, ya1, t, o[0][k], o[1][k], o[2][k]);
                if constexpr (kU8Out) {
                    // R0 G0 B0 R1 | G1 B1 R2 G2 | B2 R3 G3 B3
                    auto u = [&](int c, int k) { return __float_as_uint(o[c][k]); };
                    const uint32_t w0 = u(0, 0) | (u(1, 0) << 8) | (u(2, 0) << 16) | (u(0, 1) << 24);
                    const uint32_t w1 = u(1, 1) | (u(2, 1) << 8) | (u(0, 2) << 16) | (u(1, 2) << 24);
                    const uint32_t w2 = u(2, 2) | (u(0, 3) << 8) | (u(1, 3) << 16) | (u(2, 3) << 24);
                    __stcs(reinterpret_cast<uint32_t*>(p), w0);
                    __stcs(reinterpret_cast<uint32_t*>(p) + 1, w1);
                    __stcs(reinterpret_cast<uint32_t*>(p) + 2, w2);
                } else {
                    __stcs(reinterpret_cast<float4*>(p), make_float4(o[0][0], o[0][1], o[0][2], o[0][3]));
                    __stcs(reinterpret_cast<float4*>(const_cast<char*>(wide_imm<16>(p, plane4))), make_float4(o[1][0], o[1][1], o[1][2], o[1][3]));
                    __stcs(reinterpret_cast<float4*>(const_cast<char*>(wide_imm<32>(p, plane4))), make_float4(o[2][0], o[2][1], o[2][2], o[2][3]));
                }
            };

            // three register sets, loads two rows ahead of their use: the ncu source view of the one-row-ahead version
            // still had 47 % of its stall samples on the first use of the Lab words (load-to-use > 1.5 us behind the
            // kernel's own 12 B/px store stream)
            int y = y0 + lr;
            uint32_t al = 0, aa = 0, ab = 0, bl = 0, ba = 0, bb = 0, cl = 0, ca = 0, cb = 0;
            if (y < y1) load3(pl, al, aa, ab);
            if (y + rpi < y1) load3(wide_imm<4>(pl, step4), bl, ba, bb);
            while (y < y1) {
                if (y + 2 * rpi < y1) load3(wide_imm<8>(pl, step4), cl, ca, cb);
                map_row(y, po, al, aa, ab);
                y += rpi;
                if (y >= y1) break;
                if (y + 2 * rpi < y1) load3(wide_imm<12>(pl, step4), al, aa, ab);
                map_row(y, const_cast<char*>(wide_imm<kOB>(po, step4)), bl, ba, bb);
                y += rpi;
                if (y >= y1) break;
                if (y + 2 * rpi < y1) load3(wide_imm<16>(pl, step4), bl, ba, bb);
                map_row(y, const_cast<char*>(wide_imm<2 * kOB>(po, step4)), cl, ca, cb);
                y += rpi;
                pl = wide_imm<12>(pl, step4);
                po = const_cast<char*>(wide_imm<3 * kOB>(po, step4));
            }
        }
        __syncthreads();
        cur = nxt;
    }
    (void)sixteen;
}

// ---------------------------------------------------------------------------------------------
// K3 generic path: one thread per pixel, LUTs read through L1/L2.
// ---------------------------------------------------------------------------------------------
template <bool kU8Out>
__global__ void __launch_bounds__(256)
k_map_generic(const uint8_t* __restrict__ lab, const uint8_t* __restrict__ lut_g, void* __restrict__ out,
              int h, int w, int tiles_x, int tiles_y, float inv_tw, float inv_th)
{
    __shared__ uint32_t s_yf[256];
    __shared__ __align__(16) float s_outf[4096];
    const int tid = threadIdx.x;
    s_yf[tid] = d_labyf[tid];
    for (int i = tid; i < 1024; i += 256) reinterpret_cast<uint4*>(s_outf)[i] = reinterpret_cast<const uint4*>(d_outf_bits)[i];
    __syncthreads();

    const int f = blockIdx.y;
    const size_t plane = size_t(h) * w;
    const uint8_t* labL = lab + size_t(f) * 3 * plane;
    const uint8_t* lf = lut_g + size_t(f) * tiles_x * tiles_y * 256;
    float* outR = reinterpret_cast<float*>(out) + size_t(f) * 3 * plane;
    uint8_t* out8 = reinterpret_cast<uint8_t*>(out) + size_t(f) * 3 * plane;   // kU8Out: packed RGB (HWC)
    const uint64_t pol_stream = policy_evict_first();
    for (size_t p = size_t(blockIdx.x) * 256 + tid; p < plane; p += size_t(gridDim.x) * 256) {
        const int y = int(p / w), x = int(p - size_t(y) * w);
        const float txf = __fadd_rn(__fmul_rn(float(x), inv_tw), -0.5f);
        const float tyf = __fadd_rn(__fmul_rn(float(y), inv_th), -0.5f);
        int tx1 = __float2int_rd(txf), ty1 = __float2int_rd(tyf);
        const float xa = __fsub_rn(txf, float(tx1)), ya = __fsub_rn(tyf, float(ty1));
        const float xa1 = __fsub_rn(1.0f, xa), ya1 = __fsub_rn(1.0f, ya);
        const int tx2 = min(tx1 + 1, tiles_x - 1), ty2 = min(ty1 + 1, tiles_y - 1);
        tx1 = max(tx1, 0);
        ty1 = max(ty1, 0);
        const int v = labL[p];
        const float l11 = float(__ldg(lf + (ty1 * tiles_x + tx1) * 256 + v));
        const float l12 = float(__ldg(lf + (ty1 * tiles_x + tx2) * 256 + v));
        const float l21 = float(__ldg(lf + (ty2 * tiles_x + tx1) * 256 + v));
        const float l22 = float(__ldg(lf + (ty2 * tiles_x + tx2) * 256 + v));
        const float top = __fadd_rn(__fmul_rn(l11, xa1), __fmul_rn(l12, xa));
        const float bot = __fadd_rn(__fmul_rn(l21, xa1), __fmul_rn(l22, xa));
        const float res = __fadd_rn(__fmul_rn(top, ya1), __fmul_rn(bot, ya));
        const int Lc = min(max(__float2int_rn(res), 0), 255);
        float r, gch, b;
        lab_to_rgb_f32(Lc, labL[plane + p], labL[2 * plane + p], s_yf, s_outf, r, gch, b);
        if constexpr (kU8Out) {
            // value / 255 back to the u8 value: k / 255.f * 255.f truncates to k for every k in 0..255 (tests/test_oracle_pin.py)
            out8[3 * p + 0] = uint8_t(__float2int_rz(__fmul_rn(r, 255.0f)));
            out8[3 * p + 1] = uint8_t(__float2int_rz(__fmul_rn(gch, 255.0f)));
            out8[3 * p + 2] = uint8_t(__float2int_rz(__fmul_rn(b, 255.0f)));
        } else {
            st_stream_f1(outR + p, r, pol_stream);
            st_stream_f1(outR + plane + p, gch, pol_stream);
            st_stream_f1(outR + 2 * plane + p, b, pol_stream);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct ClaheLayout {
    size_t off_hist, off_lut, off_tickets, off_work, off_lab, total;
};

static ClaheLayout clahe_layout(int n, int h, int w, int tiles_x, int tiles_y)
{
    ClaheLayout L;
    const size_t nt = size_t(n) * tiles_x * tiles_y;
    L.off_hist = 0;
    L.off_tickets = align_up(L.off_hist + nt * 256 * sizeof(int32_t), 256);
    L.off_work = align_up(L.off_tickets + nt * sizeof(unsigned), 256);   // work-queue head of the persistent map kernel
    L.off_lut = align_up(L.off_work + 256, 256);
    L.off_lab = align_up(L.off_lut + nt * 256, 256);
    L.total = align_up(L.off_lab + size_t(n) * 3 * h * w, 256);
    return L;
}

static bool valid_shape(int n, int h, int w, int tiles_x, int tiles_y)
{
    return n >= 0 && h > 0 && w > 0 && tiles_x > 0 && tiles_y > 0 && tiles_x <= 256 && tiles_y <= 256 &&
           size_t(h) * w <= (size_t(1) << 30);
}

// cudaFuncAttributeMaxDynamicSharedMemorySize bookkeeping, one word per kernel instantiation, one bit per device ordinal.
// Written without a lock on purpose: concurrent callers can only both see "not set yet" and both issue the (idempotent)
// cudaFuncSetAttribute call; the words are atomics so that the race is a defined one.
static std::atomic<unsigned long long> g_smem_mask[4];

// storage dtypes (UPR_DT_*) and flags of the Retinex maps of a fused call; valid_map_dtypes() holds
struct MapDtypes {
    int illu = UPR_DT_F32, e = UPR_DT_F32, flags = 0;
};
static size_t map_bytes(int dt) { return dt == UPR_DT_F32 ? sizeof(float) : 2; }

// K1 with the fused Retinex prologue on maps (TI, TE): the vector kernel when `fast`, the generic one otherwise
template <typename TI, typename TE, bool AC>
static int k1_fused_launch(bool fast, dim3 grid, size_t smem, cudaStream_t stream, const float* in, uint8_t* lab, int32_t* hist,
                           uint8_t* lut, unsigned* tickets, const ClaheGeom& g, const RetinexIn& rx)
{
    if (fast) {
        static std::atomic<unsigned long long> smem_mask{0};   // one per instantiation, as g_smem_mask
        UPR_CUDA_TRY(ensure_dynamic_smem(k_hist_lab_vec3<false, true, TI, TE, AC>, smem, smem_mask));
        k_hist_lab_vec3<false, true, TI, TE, AC><<<grid, kK1Threads, smem, stream>>>(in, lab, hist, lut, tickets, g, rx);
    } else {
        k_hist_lab_generic<false, true, TI, TE, AC><<<grid, 256, 0, stream>>>(in, lab, hist, lut, g, rx);
    }
    return UPR_OK;
}

// raw tile coordinate of OpenCV's interpolation: floor(p * inv - 0.5f), fp32, separately rounded
static inline int raw_tile(int p, float inv)
{
    volatile float m = float(p) * inv;  // volatile: forbid host-side contraction
    volatile float t = m - 0.5f;
    return int(std::floor(t));
}

// stage_mask: bit 0 = K1 (Lab + histograms + LUTs), bit 1 = K3 (map); 3 = the whole op
// in_u8 / out_u8: the frame on that side is packed u8 RGB (HWC) instead of planar f32 (NCHW)
// rx: the fused Retinex prologue on maps of the dtypes `dt`
static int clahe_run(const void* in_v, void* out_v, int n, int h, int w, double clip_limit, int tiles_x, int tiles_y,
                     void* ws, size_t ws_bytes, cudaStream_t stream, int stage_mask = 3, const RetinexIn* rx = nullptr,
                     bool in_u8 = false, bool out_u8 = false, MapDtypes dt = {})
{
    if (!valid_shape(n, h, w, tiles_x, tiles_y)) return UPR_E_SHAPE;
    if (n == 0) return UPR_OK;
    if (!in_v || !out_v || !ws) return UPR_E_NULL;
    if (rx && in_u8) return UPR_E_PARAM;
    const float* in = static_cast<const float*>(in_v);      // valid when !in_u8
    float* out = static_cast<float*>(out_v);                // valid when !out_u8
    const size_t in_es = in_u8 ? 1 : sizeof(float), out_es = out_u8 ? 1 : sizeof(float);
    if (!(clip_limit == clip_limit)) return UPR_E_PARAM;
    const ClaheLayout lay = clahe_layout(n, h, w, tiles_x, tiles_y);
    if (ws_bytes < lay.total || (reinterpret_cast<uintptr_t>(ws) & 255u)) return UPR_E_WORKSPACE;

    auto* base = static_cast<unsigned char*>(ws);
    auto* hist = reinterpret_cast<int32_t*>(base + lay.off_hist);
    auto* tickets = reinterpret_cast<unsigned*>(base + lay.off_tickets);
    auto* work = reinterpret_cast<unsigned*>(base + lay.off_work);
    auto* lut = base + lay.off_lut;
    auto* lab = base + lay.off_lab;

    const bool padded = (w % tiles_x != 0) || (h % tiles_y != 0);
    const int wp = padded ? w + (tiles_x - w % tiles_x) : w;
    const int hp = padded ? h + (tiles_y - h % tiles_y) : h;

    ClaheGeom g{};
    g.n = n; g.h = h; g.w = w; g.tiles_x = tiles_x; g.tiles_y = tiles_y;
    g.tw = wp / tiles_x; g.th = hp / tiles_y;
    const int area = g.tw * g.th;
    g.clip = 0;
    if (clip_limit > 0.0) g.clip = std::max(int(clip_limit * area / 256), 1);
    g.lut_scale = float(255) / float(area);
    g.gam_bias = 0u - 4u * 0x4B000000u;
    const float inv_tw = 1.0f / float(g.tw), inv_th = 1.0f / float(g.th);

    // interpolation cell boundaries from the exact fp32 recipe (monotone in p)
    MapGeom m{};
    // (a one-row strip of a tile must fit the byte counters: <= 63 four-pixel items per thread, i.e. tiles <= 64512 px wide)
    bool fast = !padded && tiles_x <= kMaxTiles && tiles_y <= kMaxTiles && (g.tw % 4 == 0) && g.tw / 4 <= 63 * kK1Threads &&
                (in_u8 ? (reinterpret_cast<uintptr_t>(in_v) & 3u) == 0 : aligned16(in_v)) &&
                (out_u8 ? (reinterpret_cast<uintptr_t>(out_v) & 3u) == 0 : aligned16(out_v)) &&
                size_t(h) * w * 3 < (size_t(1) << 32) &&
                (!rx || ((reinterpret_cast<uintptr_t>(rx->illu) & (4 * map_bytes(dt.illu) - 1)) == 0 &&
                         (reinterpret_cast<uintptr_t>(rx->e) & (4 * map_bytes(dt.e) - 1)) == 0));   // 4 pixels of each map
    if (fast) {
        m.ay_bias = 0u - 0x4B400000u * 128u;
        m.n = n; m.h = h; m.w = w; m.tiles_x = tiles_x; m.tiles_y = tiles_y; m.inv_tw = inv_tw; m.inv_th = inv_th;
        int c = 0;
        m.bx[0] = 0;
        for (int x = 0; x < w; ++x) {
            const int t = raw_tile(x, inv_tw) + 1;  // cell index
            if (t < c || t > tiles_x) { fast = false; break; }
            while (c < t) m.bx[++c] = x;
        }
        while (c < tiles_x + 1) m.bx[++c] = w;
        c = 0;
        m.by[0] = 0;
        for (int y = 0; y < h && fast; ++y) {
            const int t = raw_tile(y, inv_th) + 1;
            if (t < c || t > tiles_y) { fast = false; break; }
            while (c < t) m.by[++c] = y;
        }
        while (c < tiles_y + 1) m.by[++c] = h;
        for (int i = 0; i <= tiles_x + 1 && fast; ++i) fast = (m.bx[i] % 4 == 0);
        if (fast) {
            const int nc = (tiles_x + 1) * (tiles_y + 1);
            long long area[(kMaxTiles + 1) * (kMaxTiles + 1)], amax = 0;
            for (int c = 0; c < nc; ++c) {
                const int cy = c / (tiles_x + 1), cx = c % (tiles_x + 1);
                area[c] = (long long)(m.bx[cx + 1] - m.bx[cx]) * (m.by[cy + 1] - m.by[cy]);
                amax = std::max(amax, area[c]);
                m.order[c] = (unsigned short)c;
            }
            std::stable_sort(m.order, m.order + nc, [&](unsigned short a, unsigned short b) { return area[a] > area[b]; });
            m.n_class[0] = m.n_class[1] = m.n_class[2] = 0;
            for (int k = 0; k < nc; ++k) {
                const long long a = area[m.order[k]];
                ++m.n_class[4 * a >= 3 * amax ? 0 : (10 * a >= 3 * amax ? 1 : 2)];
            }
        }
    }

    const int ntiles = tiles_x * tiles_y;
    // a frame index rides in gridDim.y (<= 65535): run long batches in slices
    for (int f0 = 0; f0 < n; f0 += 65535) {
        const int nf = std::min(n - f0, 65535);
        const size_t fplane = size_t(f0) * 3 * h * w;
        const size_t ftile = size_t(f0) * ntiles;
        const RetinexIn rxf = rx ? RetinexIn{static_cast<const char*>(rx->illu) + size_t(f0) * h * w * map_bytes(dt.illu),
                                             static_cast<const char*>(rx->e) + fplane * map_bytes(dt.e), rx->eps}
                                 : RetinexIn{nullptr, nullptr, 0.0f};
        auto k1_fused = [&](bool vec, dim3 grid1, size_t smem1) {
            return with_map_types(dt.illu, dt.e, dt.flags, [&](auto ti, auto te, auto ac) {
                return k1_fused_launch<typename decltype(ti)::type, typename decltype(te)::type, decltype(ac)::value>(
                    vec, grid1, smem1, stream, in + fplane, lab + fplane, hist + ftile * 256, lut + ftile * 256, tickets + ftile, g, rxf);
            });
        };
        if (fast) {
            // K1: byte counters allow <= 255 pixels per thread between flushes -> <= 63 items/thread
            const int tw4 = g.tw / 4;
            // (63 iterations of kK1Threads / tw4 rows; tiles wider than 1024 px: 63 / passes rows, one row per iteration)
            const int passes = (tw4 + kK1Threads - 1) / kK1Threads;
            const int max_rows = tw4 <= kK1Threads ? 63 * (kK1Threads / tw4) : std::max(1, 63 / passes);
            int nstrips = (g.th + max_rows - 1) / max_rows;
            const int want = (3 * kNumSMsB200 + nf * ntiles - 1) / (nf * ntiles);  // fill the machine for tiny batches
            nstrips = std::min(std::max(nstrips, want), g.th);
            g.strip_rows = (g.th + nstrips - 1) / nstrips;
            g.nstrips = (g.th + g.strip_rows - 1) / g.strip_rows;
            bool work_cleared = false;
            if (g.nstrips > 1 && (stage_mask & 1)) {
                if (f0 == 0 && nf == n && stage_mask == 3) {
                    // small batches (strips): histograms, tickets and the map kernel's queue head are adjacent in the workspace --
                    // ONE memset node instead of three (a single 1080p frame is a 50 us call: every stream operation counts)
                    UPR_CUDA_TRY(cudaMemsetAsync(base + lay.off_hist, 0, lay.off_work + sizeof(unsigned) - lay.off_hist, stream));
                    work_cleared = true;
                } else {
                    UPR_CUDA_TRY(cudaMemsetAsync(hist + ftile * 256, 0, size_t(nf) * ntiles * 256 * sizeof(int32_t), stream));
                    UPR_CUDA_TRY(cudaMemsetAsync(tickets + ftile, 0, size_t(nf) * ntiles * sizeof(unsigned), stream));
                }
            }
            const size_t smem1 = size_t(256) * kK1Threads + UPR_TAB_GAMMA_LEN * 4 + UPR_TAB_CBRT_LEN * 2;
            if (stage_mask & 1) {
                const dim3 grid1(ntiles * g.nstrips, nf);
                if (in_u8) {
                    UPR_CUDA_TRY(ensure_dynamic_smem(k_hist_lab_vec3<true, false>, smem1, g_smem_mask[0]));
                    k_hist_lab_vec3<true, false><<<grid1, kK1Threads, smem1, stream>>>(
                        static_cast<const uint8_t*>(in_v) + fplane, lab + fplane, hist + ftile * 256, lut + ftile * 256, tickets + ftile, g, rxf);
                } else if (rx) {
                    const int rc = k1_fused(true, grid1, smem1);
                    if (rc != UPR_OK) return rc;
                } else {
                    UPR_CUDA_TRY(ensure_dynamic_smem(k_hist_lab_vec3<false, false>, smem1, g_smem_mask[1]));
                    k_hist_lab_vec3<false, false><<<grid1, kK1Threads, smem1, stream>>>(
                        in + fplane, lab + fplane, hist + ftile * 256, lut + ftile * 256, tickets + ftile, g, rxf);
                }
                UPR_LAUNCH_CHECK();
            }
            const int ncells = (tiles_x + 1) * (tiles_y + 1);
            const int cell_rows = g.th;  // interior cells are one tile high
            if (stage_mask & 2) {
                {
                    // thread count: the largest multiple of the interior cell width (in 4-px columns) <= 512
                    const int cw4 = g.tw / 4;
                    int nthr = cw4 <= kK5MaxThreads ? (kK5MaxThreads / cw4) * cw4 : kK5MaxThreads;
                    if (nthr < 256) nthr = kK5MaxThreads;
                    const size_t smem5 = size_t(kXzLinBytes) + 4096 * 4 + 512 * 4 * 16 + 2 * 256 * 4;
                    // items = (frame, cell, strip): ~4 items per resident CTA on small batches, strips of >= 16 rows (every item
                    // costs a barrier and a quad-table build: with 16 items per CTA and 8-row strips a 3-frame call took 99 us
                    // instead of 78 us for a one-CTA-per-item kernel)
                    const int resident = 2 * kNumSMsB200;
                    int ks5 = std::max(1, int((size_t(4) * resident + size_t(nf) * ncells - 1) / (size_t(nf) * ncells)));
                    ks5 = std::min(ks5, std::max(cell_rows / 16, 1));
                    m.nstrips = ks5;
                    m.n = nf;          // frames of THIS launch: the queue order interleaves them (map_item)
                    const long long nitems = (long long)nf * ncells * ks5;
                    if (nitems > 0x7fffffffLL / 2) return UPR_E_SHAPE;
                    if (!work_cleared) UPR_CUDA_TRY(cudaMemsetAsync(work, 0, sizeof(unsigned), stream));
                    const dim3 grid5(unsigned(std::min<long long>(nitems, resident)));
                    void* outf = static_cast<char*>(out_v) + fplane * out_es;
                    if (out_u8) {
                        UPR_CUDA_TRY(ensure_dynamic_smem(k_map_vec5<true, true>, smem5, g_smem_mask[2]));
                        k_map_vec5<true, true><<<grid5, nthr, smem5, stream>>>(lab + fplane, lut + ftile * 256, outf, m, work, int(nitems));
                    } else {
                        UPR_CUDA_TRY(ensure_dynamic_smem(k_map_vec5<true, false>, smem5, g_smem_mask[3]));
                        k_map_vec5<true, false><<<grid5, nthr, smem5, stream>>>(lab + fplane, lut + ftile * 256, outf, m, work, int(nitems));
                    }
                }
                UPR_LAUNCH_CHECK();
            }
        } else {
            g.nstrips = 1; g.strip_rows = g.th;
            if (stage_mask & 1) {
                const void* inf = static_cast<const char*>(in_v) + fplane * in_es;
                const dim3 grid1(ntiles, nf);
                if (in_u8) k_hist_lab_generic<true, false><<<grid1, 256, 0, stream>>>(inf, lab + fplane, hist + ftile * 256, lut + ftile * 256, g, rxf);
                else if (rx) {
                    const int rc = k1_fused(false, grid1, 0);
                    if (rc != UPR_OK) return rc;
                } else k_hist_lab_generic<false, false><<<grid1, 256, 0, stream>>>(inf, lab + fplane, hist + ftile * 256, lut + ftile * 256, g, rxf);
                UPR_LAUNCH_CHECK();
            }
            const size_t plane = size_t(h) * w;
            const int gx = int(std::min<size_t>((plane + 255) / 256, 4096));
            if (stage_mask & 2) {
                void* outf = static_cast<char*>(out_v) + fplane * out_es;
                if (out_u8) k_map_generic<true><<<dim3(gx, nf), 256, 0, stream>>>(lab + fplane, lut + ftile * 256, outf, h, w, tiles_x, tiles_y, inv_tw, inv_th);
                else k_map_generic<false><<<dim3(gx, nf), 256, 0, stream>>>(lab + fplane, lut + ftile * 256, outf, h, w, tiles_x, tiles_y, inv_tw, inv_th);
                UPR_LAUNCH_CHECK();
            }
        }
    }
    return UPR_OK;
}

}  // namespace upr

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

size_t upr_clahe_workspace_bytes(int n, int h, int w, int tiles_x, int tiles_y)
{
    if (!upr::valid_shape(n, h, w, tiles_x, tiles_y)) return 0;
    return upr::clahe_layout(std::max(n, 1), h, w, tiles_x, tiles_y).total;
}

int upr_clahe_lab_f32(const float* in_nchw, float* out_nchw, int n, int h, int w, double clip_limit, int tiles_x,
                      int tiles_y, void* workspace, size_t workspace_bytes, upr_stream_t stream)
{
    return upr::clahe_run(in_nchw, out_nchw, n, h, w, clip_limit, tiles_x, tiles_y, workspace, workspace_bytes,
                          static_cast<cudaStream_t>(stream));
}

int upr_retinex_clahe_f32(const float* x, const float* illu, const float* e, float* out_nchw, int n, int h, int w, float eps,
                          double clip_limit, int tiles_x, int tiles_y, void* workspace, size_t workspace_bytes,
                          upr_stream_t stream)
{
    if (!x || !illu || !e) return (n == 0 && upr::valid_shape(n, h, w, tiles_x, tiles_y)) ? UPR_OK : UPR_E_NULL;
    const upr::RetinexIn rx{illu, e, eps};
    return upr::clahe_run(x, out_nchw, n, h, w, clip_limit, tiles_x, tiles_y, workspace, workspace_bytes,
                          static_cast<cudaStream_t>(stream), 3, &rx);
}

int upr_retinex_clahe_f32_u8(const float* x, const float* illu, const float* e, unsigned char* out_nhwc, int n, int h, int w,
                             float eps, double clip_limit, int tiles_x, int tiles_y, void* workspace, size_t workspace_bytes,
                             upr_stream_t stream)
{
    if (!x || !illu || !e) return (n == 0 && upr::valid_shape(n, h, w, tiles_x, tiles_y)) ? UPR_OK : UPR_E_NULL;
    const upr::RetinexIn rx{illu, e, eps};
    return upr::clahe_run(x, out_nhwc, n, h, w, clip_limit, tiles_x, tiles_y, workspace, workspace_bytes,
                          static_cast<cudaStream_t>(stream), 3, &rx, false, true);
}

// the typed entries: the checks of the f32 ones (shape, then the dtypes and flags, then n == 0, then NULL) before clahe_run
static int retinex_clahe_typed(const float* x, const void* illu, int illu_dtype, const void* e, int e_dtype, int flags, void* out,
                               bool out_u8, int n, int h, int w, float eps, double clip_limit, int tiles_x, int tiles_y,
                               void* workspace, size_t workspace_bytes, cudaStream_t stream)
{
    if (!upr::valid_shape(n, h, w, tiles_x, tiles_y)) return UPR_E_SHAPE;
    if (!upr::valid_map_dtypes(illu_dtype, e_dtype, flags)) return UPR_E_PARAM;
    if (n == 0) return UPR_OK;
    if (!x || !illu || !e) return UPR_E_NULL;
    const upr::RetinexIn rx{illu, e, eps};
    upr::MapDtypes dt;
    dt.illu = illu_dtype;
    dt.e = e_dtype;
    dt.flags = flags;
    return upr::clahe_run(x, out, n, h, w, clip_limit, tiles_x, tiles_y, workspace, workspace_bytes, stream, 3, &rx, false, out_u8,
                          dt);
}

int upr_retinex_clahe_typed_f32(const float* x, const void* illu, int illu_dtype, const void* e, int e_dtype, int flags,
                                float* out_nchw, int n, int h, int w, float eps, double clip_limit, int tiles_x, int tiles_y,
                                void* workspace, size_t workspace_bytes, upr_stream_t stream)
{
    return retinex_clahe_typed(x, illu, illu_dtype, e, e_dtype, flags, out_nchw, false, n, h, w, eps, clip_limit, tiles_x, tiles_y,
                               workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int upr_retinex_clahe_typed_u8(const float* x, const void* illu, int illu_dtype, const void* e, int e_dtype, int flags,
                               unsigned char* out_nhwc_rgb, int n, int h, int w, float eps, double clip_limit, int tiles_x,
                               int tiles_y, void* workspace, size_t workspace_bytes, upr_stream_t stream)
{
    return retinex_clahe_typed(x, illu, illu_dtype, e, e_dtype, flags, out_nhwc_rgb, true, n, h, w, eps, clip_limit, tiles_x,
                               tiles_y, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int upr_clahe_lab_u8(const unsigned char* in_nhwc, unsigned char* out_nhwc, int n, int h, int w, double clip_limit, int tiles_x,
                     int tiles_y, void* workspace, size_t workspace_bytes, upr_stream_t stream)
{
    return upr::clahe_run(in_nhwc, out_nhwc, n, h, w, clip_limit, tiles_x, tiles_y, workspace, workspace_bytes,
                          static_cast<cudaStream_t>(stream), 3, nullptr, true, true);
}

int upr_clahe_lab_f32_u8(const float* in_nchw, unsigned char* out_nhwc, int n, int h, int w, double clip_limit, int tiles_x,
                         int tiles_y, void* workspace, size_t workspace_bytes, upr_stream_t stream)
{
    return upr::clahe_run(in_nchw, out_nhwc, n, h, w, clip_limit, tiles_x, tiles_y, workspace, workspace_bytes,
                          static_cast<cudaStream_t>(stream), 3, nullptr, false, true);
}

int upr_clahe_lab_stages_f32(const float* in_nchw, float* out_nchw, int n, int h, int w, double clip_limit, int tiles_x,
                             int tiles_y, void* workspace, size_t workspace_bytes, int stage_mask, upr_stream_t stream)
{
    if ((stage_mask & 3) == 0) return UPR_E_PARAM;
    return upr::clahe_run(in_nchw, out_nchw, n, h, w, clip_limit, tiles_x, tiles_y, workspace, workspace_bytes,
                          static_cast<cudaStream_t>(stream), stage_mask & 3);
}

int upr_clahe_debug_dump(const void* workspace, int n, int h, int w, int tiles_x, int tiles_y, int32_t* hist_out,
                         uint8_t* lut_out, uint8_t* lab_out, upr_stream_t stream)
{
    if (!upr::valid_shape(n, h, w, tiles_x, tiles_y)) return UPR_E_SHAPE;
    if (!workspace) return UPR_E_NULL;
    if (n == 0) return UPR_OK;
    const upr::ClaheLayout lay = upr::clahe_layout(n, h, w, tiles_x, tiles_y);
    const auto* base = static_cast<const unsigned char*>(workspace);
    auto s = static_cast<cudaStream_t>(stream);
    const size_t nt = size_t(n) * tiles_x * tiles_y;
    if (hist_out) UPR_CUDA_TRY(cudaMemcpyAsync(hist_out, base + lay.off_hist, nt * 256 * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
    if (lut_out) UPR_CUDA_TRY(cudaMemcpyAsync(lut_out, base + lay.off_lut, nt * 256, cudaMemcpyDeviceToDevice, s));
    if (lab_out) UPR_CUDA_TRY(cudaMemcpyAsync(lab_out, base + lay.off_lab, size_t(n) * 3 * h * w, cudaMemcpyDeviceToDevice, s));
    return UPR_OK;
}

int upr_clahe_debug_load(void* workspace, int n, int h, int w, int tiles_x, int tiles_y, const uint8_t* lut_in,
                         const uint8_t* lab_in, upr_stream_t stream)
{
    if (!upr::valid_shape(n, h, w, tiles_x, tiles_y)) return UPR_E_SHAPE;
    if (!workspace) return UPR_E_NULL;
    if (n == 0) return UPR_OK;
    const upr::ClaheLayout lay = upr::clahe_layout(n, h, w, tiles_x, tiles_y);
    auto* base = static_cast<unsigned char*>(workspace);
    auto s = static_cast<cudaStream_t>(stream);
    const size_t nt = size_t(n) * tiles_x * tiles_y;
    if (lut_in) UPR_CUDA_TRY(cudaMemcpyAsync(base + lay.off_lut, lut_in, nt * 256, cudaMemcpyDeviceToDevice, s));
    if (lab_in) UPR_CUDA_TRY(cudaMemcpyAsync(base + lay.off_lab, lab_in, size_t(n) * 3 * h * w, cudaMemcpyDeviceToDevice, s));
    return UPR_OK;
}

int upr_get_tables(uint16_t* gamma, uint16_t* cbrt, uint32_t* labyf, uint8_t* invgamma)
{
    if (gamma) std::memcpy(gamma, upr::h_gamma, sizeof upr::h_gamma);
    if (cbrt) std::memcpy(cbrt, upr::h_cbrt, sizeof upr::h_cbrt);
    if (labyf) std::memcpy(labyf, upr::h_labyf, sizeof upr::h_labyf);
    if (invgamma) std::memcpy(invgamma, upr::h_invgamma, sizeof upr::h_invgamma);
    return UPR_OK;
}

}  // extern "C"
