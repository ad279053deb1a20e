// Shared pieces of the ROI-crop translation units (crop.cu: prep, per-strip and generic kernels, entry points; crop_cta.cu: the
// warp-specialised one-crop-per-CTA kernel): geometry record, tap arithmetic of cv2.resize(INTER_AREA) (SURVEY.md App. C),
// output writers, the bit-exact horizontal passes and the TMA / mbarrier wrappers.
#pragma once
#include <cuda.h>

#include <stdlib.h>

#include <type_traits>

#include "common.cuh"

namespace bpc {

constexpr int CROP_BAND = 8;                 // generic kernel: output rows per work item
constexpr int CROP_RAW_BYTES = 40 * 1024;    // generic kernel: staged source bytes
constexpr int WARP_BUF = 3584;               // warp kernel: bytes of one staging buffer (two per warp)
constexpr int WARP_DESC = 32 * 16;           // warp kernel: 32 row descriptors (two rings per warp)
constexpr int WARP_SMEM = 8320;              // 2 staging buffers + 2 descriptor rings + eight mbarriers, padded to a multiple of 128
static_assert(WARP_SMEM % 128 == 0 && WARP_SMEM >= 2 * WARP_BUF + 2 * WARP_DESC + 64 && WARP_BUF % 128 == 0, "TMA box destinations are 128-byte aligned");
constexpr int WARPK_WARPS = 8;
constexpr int LUT_STRIDE = 257;              // shared-memory LUT: 256 entries + the normalised fill value per output channel
constexpr int LUT_SMEM = 3200;               // 3 * 257 floats, padded to a multiple of 128 (TMA destinations follow)
constexpr int WARPK_SMEM = WARPK_WARPS * WARP_SMEM + LUT_SMEM;
constexpr int CTA_ROWS = 8;                  // CTA kernel: source rows per ring slot (= one TMA box); per-source-row records come in whole slots
constexpr int YSRC_PAD = 16;                 // per-source-row table: zero entries behind the last row (whole slots run to completion)
static_assert(LUT_SMEM % 128 == 0 && LUT_SMEM >= 3 * LUT_STRIDE * 4, "LUT block");
// descriptors per ROI: x axis ds float4, y axis ds + 8 float4 (class 1 reads the y block as 2*ds + 16 float2 source-row records),
// ds = T rounded up to 32
__host__ __device__ __forceinline__ int desc_stride(int T) { return (T + 31) & ~31; }
// float4 records per ROI on the y axis: ds + 8 (class 1 reads the block as 2 ds + 16 float2 source-row records); up to T = 256 the
// block also holds the source-row records of a class-4 crop for the CTA kernel (h <= 5 T rows + one padded slot + 16)
__host__ __device__ __forceinline__ int ydesc_stride(int T) {
    const int base = desc_stride(T) + 8, rows4 = (5 * T + 32 + 1) / 2;
    return (T <= 256 && rows4 > base) ? rows4 : base;
}

struct RoiGeom {                             // 88 bytes, workspace
    double scale_x, scale_y, inv_x, inv_y;
    unsigned long long src;                  // byte address of (y1, x1) in its image
    int w, h, new_w, new_h, dx, dy;
    int regime;                              // 0 rejected, 1 / 2 / 3
    int cls;                                 // -1 beyond the device count, 0 rejected (all fill), 1 fast area, 3 fast linear, 2 generic
    int isx, isy;
    int pitch, pad_;
};
static_assert(sizeof(RoiGeom) == 88, "RoiGeom layout");

// L2 promotion of the CTA kernel's tensor maps (crop_cta.cu)
#ifndef BPC_L2_PROMO
#define BPC_L2_PROMO CU_TENSOR_MAP_L2_PROMOTION_L2_128B
#endif
// Widest staging row of a class-4 strip on the warp kernel (four ring slots of at least three rows fit 2 * WARP_BUF); the CTA
// kernel takes only pools whose row pitch is at least this wide
constexpr int WARP_MAX_PITCH = 576;

struct YDesc {                               // generic kernel, per output row of the band
    int start;
    int n;                                   // taps (regime 1/2) ; regime 3: second source row
    float bf, bm, bl;                        // regime 1 weights ; regime 3: b0, b1 as int bits
    int flags;                               // bit0 has_first, bit1 has_last
};

__device__ __forceinline__ uint4 ld_nc_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// computeResizeAreaTab for one destination index d (OpenCV resize.cpp), all in float64.
__device__ __forceinline__ void area_taps(int d, double scale, int ssize, int& start, int& n, float& af, float& am, float& al, int& flags) {
    const double fsx1 = dmul((double)d, scale);
    const double fsx2 = dadd(fsx1, scale);
    const double cell = fmin(scale, dsub((double)ssize, fsx1));
    int sx1 = (int)ceil(fsx1), sx2 = (int)floor(fsx2);
    sx2 = min(sx2, ssize - 1);
    sx1 = min(sx1, sx2);
    flags = 0;
    af = 0.f; al = 0.f;
    am = __double2float_rn(ddiv(1.0, cell));
    start = sx1;
    n = sx2 - sx1;
    if (dsub((double)sx1, fsx1) > 1e-3) {
        flags |= 1;
        af = __double2float_rn(ddiv(dsub((double)sx1, fsx1), cell));
        start = sx1 - 1;
        ++n;
    }
    if (dsub(fsx2, (double)sx2) > 1e-3) {
        flags |= 2;
        al = __double2float_rn(ddiv(fmin(fmin(dsub(fsx2, (double)sx2), 1.0), cell), cell));
        ++n;
    }
}

// index of the last source tap of destination index d: start + n - 1 of area_taps() = sx2 - 1 + (the last-tap test), without
// the weights (no divisions)
__device__ __forceinline__ int area_last_tap(int d, double scale, int ssize) {
    const double fsx2 = dadd(dmul((double)d, scale), scale);
    const int sx2 = min((int)floor(fsx2), ssize - 1);
    return sx2 - 1 + (dsub(fsx2, (double)sx2) > 1e-3 ? 1 : 0);
}

// the same taps as a start index and three weights (absent taps = +0.0f); valid when n <= 3 (scale < 2)
__device__ __forceinline__ void area_taps3(int d, double scale, int ssize, int& start, int& n, float& w0, float& w1, float& w2) {
    float af, am, al;
    int flags;
    area_taps(d, scale, ssize, start, n, af, am, al, flags);
    float w[3] = {0.f, 0.f, 0.f};
    int k = 0;
    if (flags & 1) w[k++] = af;
    const int m = n - (flags & 1) - ((flags >> 1) & 1);
    for (int t = 0; t < m && k < 3; ++t) w[k++] = am;
    if ((flags & 2) && k < 3) w[k++] = al;
    w0 = w[0]; w1 = w[1]; w2 = w[2];
}

// area-mode coordinates of the generic linear resize for one destination index d.
__device__ __forceinline__ void linear_coef(int d, double scale, double inv, int ssize, int& s0, int& w0, int& w1, int& edge) {
    int s = (int)floor(dmul((double)d, scale));
    float f = __double2float_rn(dsub((double)(d + 1), dmul((double)(s + 1), inv)));
    f = (f <= 0.f) ? 0.f : __fsub_rn(f, floorf(f));
    if (s < 0) { f = 0.f; s = 0; }
    edge = 0;
    if (s + 1 >= ssize) {
        edge = 1;
        if (s >= ssize - 1) { f = 0.f; s = ssize - 1; }
    }
    s0 = s;
    w0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f));
    w1 = __float2int_rn(__fmul_rn(f, 2048.f));
}


// ------------------------------------------------------------------------------------------------------
// shared output helpers
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned short bf16_bits(float v) {       // round-to-nearest-even float32 -> bfloat16
    unsigned short r;
    asm("cvt.rn.bf16.f32 %0, %1;" : "=h"(r) : "f"(v));
    return r;
}

// BF16: the float path's values rounded to bfloat16 and stored channels-last ([R][T][T][3], what a bf16 tensor-core network reads)
template <bool OUT_U8, bool BF16 = false>
struct Out {
    float* outf; uint8_t* outb;
    const float* lut;           // shared memory [3][LUT_STRIDE]
    int T, swap_rb;
    uint8_t fillc[3];
    float padf[3];

    __device__ __forceinline__ void px(int roi, int y, int x, int b0, int b1, int b2) const {   // source channel order
        if (OUT_U8) {
            uint8_t* o = outb + (((size_t)roi * T + y) * T + x) * 3;
            o[0] = (uint8_t)b0; o[1] = (uint8_t)b1; o[2] = (uint8_t)b2;
        } else {
            const int s0 = swap_rb ? b2 : b0, s2 = swap_rb ? b0 : b2;
            if (BF16) {
                unsigned short* o = reinterpret_cast<unsigned short*>(outf) + (((size_t)roi * T + y) * T + x) * 3;
                o[0] = bf16_bits(lut[s0]); o[1] = bf16_bits(lut[LUT_STRIDE + b1]); o[2] = bf16_bits(lut[2 * LUT_STRIDE + s2]);
            } else {
                float* o = outf + ((size_t)roi * 3 * T + y) * T + x;
                o[0] = lut[s0];
                o[(size_t)T * T] = lut[LUT_STRIDE + b1];
                o[(size_t)2 * T * T] = lut[2 * LUT_STRIDE + s2];
            }
        }
    }
    __device__ __forceinline__ void pad(int roi, int y, int x) const {
        if (OUT_U8) {
            uint8_t* o = outb + (((size_t)roi * T + y) * T + x) * 3;
            o[0] = fillc[0]; o[1] = fillc[1]; o[2] = fillc[2];
        } else if (BF16) {
            unsigned short* o = reinterpret_cast<unsigned short*>(outf) + (((size_t)roi * T + y) * T + x) * 3;
            o[0] = bf16_bits(padf[0]); o[1] = bf16_bits(padf[1]); o[2] = bf16_bits(padf[2]);
        } else {
            float* o = outf + ((size_t)roi * 3 * T + y) * T + x;
            o[0] = padf[0]; o[(size_t)T * T] = padf[1]; o[(size_t)2 * T * T] = padf[2];
        }
    }
    // rows [ra, rb) of all three planes = fill; collective over nth threads
    __device__ void pad_rows(int roi, int ra, int rb, int tid, int nth) const {
        if (rb <= ra) return;
        if (OUT_U8) {
            uint8_t* o = outb + ((size_t)roi * T + ra) * T * 3;
            const int nbytes = (rb - ra) * T * 3;
            for (int e = tid; e < nbytes; e += nth) o[e] = fillc[e % 3];
        } else if (BF16) {
            unsigned short* o = reinterpret_cast<unsigned short*>(outf) + ((size_t)roi * T + ra) * T * 3;
            const int n = (rb - ra) * T * 3;
            const unsigned short f0 = bf16_bits(padf[0]), f1 = bf16_bits(padf[1]), f2 = bf16_bits(padf[2]);
            if ((((size_t)(uintptr_t)o) & 3) == 0 && (n & 1) == 0) {          // 32-bit stores of the period-3 pattern
                unsigned* o2 = reinterpret_cast<unsigned*>(o);
                const unsigned p0 = f0 | ((unsigned)f1 << 16), p1 = f2 | ((unsigned)f0 << 16), p2 = f1 | ((unsigned)f2 << 16);
                for (int e = tid; e < (n >> 1); e += nth) { const int m = e % 3; o2[e] = m == 0 ? p0 : (m == 1 ? p1 : p2); }
            } else {
                for (int e = tid; e < n; e += nth) { const int m = e % 3; o[e] = m == 0 ? f0 : (m == 1 ? f1 : f2); }
            }
        } else if ((T & 3) == 0) {
            const int n4 = (rb - ra) * (T >> 2);
            for (int p = 0; p < 3; ++p) {
                float4* o = reinterpret_cast<float4*>(outf + ((size_t)(roi * 3 + p) * T + ra) * T);
                const float4 v = make_float4(padf[p], padf[p], padf[p], padf[p]);
                for (int e = tid; e < n4; e += nth) o[e] = v;
            }
        } else {
            const int n1 = (rb - ra) * T;
            for (int p = 0; p < 3; ++p) {
                float* o = outf + ((size_t)(roi * 3 + p) * T + ra) * T;
                for (int e = tid; e < n1; e += nth) o[e] = padf[p];
            }
        }
    }
};

template <bool OUT_U8, bool BF16>
__device__ __forceinline__ void out_init(Out<OUT_U8, BF16>& o, float* outf, uint8_t* outb, const float* lut_s, int T, int swap_rb, uchar4 fill) {
    o.outf = outf; o.outb = outb; o.lut = lut_s; o.T = T; o.swap_rb = swap_rb;
    o.fillc[0] = fill.x; o.fillc[1] = fill.y; o.fillc[2] = fill.z;
    if (!OUT_U8)
        for (int p = 0; p < 3; ++p) o.padf[p] = lut_s[p * LUT_STRIDE + o.fillc[swap_rb ? 2 - p : p]];
}


// ------------------------------------------------------------------------------------------------------
// arithmetic and staging helpers of the fast kernels
// ------------------------------------------------------------------------------------------------------
// ---- packed float32x2 arithmetic (sm_100a FFMA2 / FADD2), every lane IEEE round-to-nearest ----
typedef unsigned long long u64;
__device__ __forceinline__ u64 pack2(float lo, float hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(u64 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ u64 ffma2(u64 a, u64 b, u64 c) { u64 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ u64 fadd2(u64 a, u64 b) { u64 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
// ptxas 12.9 contracts a mul.rn.f32x2 feeding an add.rn.f32x2 into one FFMA2 (even with --fmad=false and
// volatile asm; the scalar forms are left alone): one rounding where OpenCV rounds twice, seen as 1-LSB
// errors in ~1e-4 of the pixels.  fma(a, b, -0.0) with a literal -0 is simplified back to a multiply and
// contracted again.  The vertical pass therefore forms its rounded products as fma(a, b, z) with
// z = (-0.0f, -0.0f) held in a register whose value the compiler cannot prove: the same value as a * b for
// non-negative operands, and an FFMA2 cannot be merged with the add that follows.
__device__ __forceinline__ u64 fprod2(u64 a, u64 b, u64 negzero2) { return ffma2(a, b, negzero2); }

// float(2^23 + byte K of v): the byte dropped into the mantissa of 8388608.0f (one PRMT, no I2F)
template <int K>
__device__ __forceinline__ float magic_byte(unsigned v) { return __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7540 + K)); }

// Column weights of the 3-slot horizontal pass.  fl(b * w) is computed as fma(2^23 + b, w, -(2^23 * w)):
// the product 2^23 * w is exact, so the fused result is the correctly rounded b * w, bit-identical to
// OpenCV's separately rounded multiply.
struct ColW {
    float w[3], c[3];       // weight and -(2^23 * weight) per slot
    __device__ __forceinline__ void set(float a, float b, float d) {
        w[0] = a; w[1] = b; w[2] = d;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            c[k] = __fmul_rn(w[k], -8388608.0f);
            asm volatile("" : "+f"(c[k]));      // opaque: keep it in a register instead of re-multiplying in the inner loop
        }
    }
};

// shared-memory accesses through 32-bit shared-window addresses (no generic-address arithmetic in the hot loop)
__device__ __forceinline__ unsigned lds_u32(unsigned addr) { unsigned v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }
__device__ __forceinline__ unsigned lds_u8(unsigned addr) { unsigned v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }
__device__ __forceinline__ float lds_f32(unsigned addr) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr)); return v; }
__device__ __forceinline__ float4 lds_f4(unsigned addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

// output store of the fast paths: the crop buffer is written once and never re-read by this kernel
// (-DBPC_WHATIF=1|2|3: the what-if builds behind DESIGN.md 3.2 -- one plane only / shared-memory stores / no stores)
template <int K = 0>
__device__ __forceinline__ void stg_out(float* p, float v) {
#if defined(BPC_WHATIF) && BPC_WHATIF == 1          // only plane 0 is stored
    if (K == 0) *p = v; else asm volatile("" :: "f"(v));
#elif defined(BPC_WHATIF) && BPC_WHATIF == 2        // LSU traffic without L2 traffic: the value goes to shared memory
    asm volatile("st.shared.f32 [%0], %1;" :: "r"(((unsigned)(size_t)p) & 0x7cu), "f"(v));
#elif defined(BPC_WHATIF) && BPC_WHATIF == 3        // no store, LUT value still loaded
    asm volatile("" :: "f"(v));
#elif defined(BPC_STG_CS)
    __stcs(p, v);
#else
    *p = v;
#endif
}

// horizontal pass of one source row for one output column: 9 bytes starting at shared address a4 + sh/8
__device__ __forceinline__ void h_area3(unsigned a4, int sh, const ColW& cw, u64& h01, float& h2) {
    const unsigned q0 = lds_u32(a4), q1 = lds_u32(a4 + 4), q2 = lds_u32(a4 + 8);
    const unsigned v0 = __funnelshift_r(q0, q1, sh), v1 = __funnelshift_r(q1, q2, sh), v2 = q2 >> sh;
    // pixel k = bytes 3k .. 3k+2; the (w, w) / (c, c) pairs become scalar-broadcast operands of FFMA2
    const u64 p0 = ffma2(pack2(magic_byte<0>(v0), magic_byte<1>(v0)), pack2(cw.w[0], cw.w[0]), pack2(cw.c[0], cw.c[0]));
    const u64 p1 = ffma2(pack2(magic_byte<3>(v0), magic_byte<0>(v1)), pack2(cw.w[1], cw.w[1]), pack2(cw.c[1], cw.c[1]));
    const u64 p2 = ffma2(pack2(magic_byte<2>(v1), magic_byte<3>(v1)), pack2(cw.w[2], cw.w[2]), pack2(cw.c[2], cw.c[2]));
    const float r0 = __fmaf_rn(magic_byte<2>(v0), cw.w[0], cw.c[0]);
    const float r1 = __fmaf_rn(magic_byte<1>(v1), cw.w[1], cw.c[1]);
    const float r2 = __fmaf_rn(magic_byte<0>(v2), cw.w[2], cw.c[2]);
    h01 = fadd2(fadd2(p0, p1), p2);
    h2 = __fadd_rn(__fadd_rn(r0, r1), r2);
}

// horizontal pass with NT taps evaluated (4..6): 3*NT bytes starting at shared address a4 + sh/8.  Taps beyond a
// lane's own count carry weight +0.0f (c = -0.0f): fma(2^23 + b, +0, -0) = +0 and s + (+0) = s, so padding the
// tap list to the warp's maximum leaves every sum bit-identical to the sequential ((S0*w0 + S1*w1) + ...) order.
template <int NT>
__device__ __forceinline__ void h_area_n(unsigned a4, int sh, const float (&w)[6], const float (&c)[6], u64& h01, float& h2) {
    constexpr int NV = (3 * NT + 3) / 4;            // aligned words holding 3*NT bytes; NV + 1 raw words cover any shift
    unsigned q[NV + 1], v[NV];
#pragma unroll
    for (int i = 0; i <= NV; ++i) q[i] = lds_u32(a4 + 4 * i);
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = __funnelshift_r(q[i], q[i + 1], sh);
#pragma unroll
    for (int k = 0; k < NT; ++k) {
        const int j = 3 * k;
        const float b0 = __uint_as_float(__byte_perm(v[j >> 2], 0x4B000000u, 0x7540 + (j & 3)));
        const float b1 = __uint_as_float(__byte_perm(v[(j + 1) >> 2], 0x4B000000u, 0x7540 + ((j + 1) & 3)));
        const float b2 = __uint_as_float(__byte_perm(v[(j + 2) >> 2], 0x4B000000u, 0x7540 + ((j + 2) & 3)));
        const u64 p = ffma2(pack2(b0, b1), pack2(w[k], w[k]), pack2(c[k], c[k]));
        const float r = __fmaf_rn(b2, w[k], c[k]);
        h01 = (k == 0) ? p : fadd2(h01, p);
        h2 = (k == 0) ? r : __fadd_rn(h2, r);
    }
}

// horizontal pass of the fixed-point bilinear: 6 bytes at shared address a4 + sh/8, result pre-shifted by 4
__device__ __forceinline__ void h_lin(unsigned a4, int sh, int w0, int w1, int* h) {
    const unsigned q0 = lds_u32(a4), q1 = lds_u32(a4 + 4), q2 = lds_u32(a4 + 8);
    const unsigned v0 = __funnelshift_r(q0, q1, sh), v1 = __funnelshift_r(q1, q2, sh);
    h[0] = (int)((v0 & 0xffu) * w0 + (v0 >> 24) * w1) >> 4;
    h[1] = (int)(((v0 >> 8) & 0xffu) * w0 + (v1 & 0xffu) * w1) >> 4;
    h[2] = (int)(((v0 >> 16) & 0xffu) * w0 + ((v1 >> 8) & 0xffu) * w1) >> 4;
}

// cvRound(v) for 0 <= v < 2^22 without F2I: adding 2^23 leaves round-half-even(v) in the low mantissa bits
// (no clamp: the tap weights of each axis sum to 1 within a few ulp, so v <= 255.001 and the result is <= 255)
__device__ __forceinline__ int round_u8(float v) { return __float_as_int(__fadd_rn(v, 8388608.0f)) & 0xff; }
// shared address of LUT[cvRound(v)]: lut_m = lut_base - 4 * 0x4B000000 (mod 2^32)
__device__ __forceinline__ unsigned lut_addr(float v, unsigned lut_m) { return (unsigned)__float_as_int(__fadd_rn(v, 8388608.0f)) * 4u + lut_m; }

// ---- TMA bulk copy (cp.async.bulk, SASS UBLKCP) completing on an mbarrier in shared memory ----
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, unsigned long long src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
#ifndef BPC_MBAR_HINT_NS
#define BPC_MBAR_HINT_NS 2000
#endif
// try_wait with a suspend-time hint: a waiting warp sleeps in hardware until the phase completes (or the hint elapses) instead of
// spinning through try_wait / yield / branch -- spinning consumer and producer warps executed 30 % of the CTA kernel's
// instructions before the hint was added
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "BPC_WAIT:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
                 "@p bra BPC_DONE;\n"
                 "bra BPC_WAIT;\n"
                 "BPC_DONE:\n"
                 "}" :: "r"(bar), "r"(parity), "r"((unsigned)BPC_MBAR_HINT_NS) : "memory");
}

__device__ __forceinline__ int warp_max_i32(int v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, m));
    return v;
}


// ---- the CTA kernel (crop_cta.cu) as seen from the launcher in crop.cu ----
constexpr int CTA_MAX_T = 256;               // 8 consumer warps
__host__ __device__ __forceinline__ int cta_pitch_max(int T) { return ((15 + 3 * (2 * T - 1) + 12 + 63) >> 6) << 6; }
// out_mode: 0 float32 [R][3][T][T], 1 uint8 [R][T][T][3], 2 bfloat16 [R][T][T][3]; list / counters as written by bpc_crop_prep_kernel
int crop_cta_launch(int out_mode, const uint8_t* images, int B, int H, int W, const RoiGeom* geom, const float4* xdesc, const float4* ydesc,
                    const int32_t* list1, int32_t* counters, int R, int T, uchar4 fill, int swap_rb, const float* lut, float* outf,
                    uint8_t* outb, cudaStream_t st);

}  // namespace bpc
