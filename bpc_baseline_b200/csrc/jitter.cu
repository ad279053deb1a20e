// ColorJitter of the training crops: torchvision.transforms.ColorJitter applied to Image.fromarray(canvas) of a uint8
// letterboxed crop (what BOPSingleObjDataset.__getitem__ does after the crop, bpc/utils/data_utils.py), followed by
// to_tensor + normalize through the 3 x 256 LUT -- bit-exact with Pillow's arithmetic:
//
//   blend(a, x, f)   Image.blend: float32 a + f * (x - a), multiply and add rounded separately, truncated
//                    (clipped to [0, 255] first when f is outside [0, 1])
//   brightness f     blend(0, x, f)                 -> a byte table per crop
//   contrast f       blend(mean, x, f)              -> a byte table per crop once the mean is known;
//                    mean = int(sum(L) / (T*T) + 0.5) over the image AS IT STANDS when contrast runs (ImageStat)
//   saturation f     blend(L, x, f), L = (19595 R + 38470 G + 7471 B + 0x8000) >> 16
//   hue f            RGB -> HSV (Pillow), h += uint8(int32(f * 255.0)) mod 256, HSV -> RGB (Pillow)
//
// One CTA per crop and no shared-memory copy of the image.  Phase 1 (only when contrast is enabled) streams the crop,
// applies the ops that come before contrast and block-reduces the integer L sum; phase 2 re-reads the crop (L2-resident:
// 147 KB at T=224, 197 KB at T=256; two CTAs per SM keep ~60 MB of crops in flight), applies the whole chain and writes
// the three float planes.  DRAM traffic is 3 T^2 bytes read + 12 T^2 bytes written per crop.  Before phase 2 the chain is
// compiled per crop: adjacent table ops (brightness, contrast) are composed into one byte table, and a table run at the
// end of the chain is folded into the output LUT, so brightness + contrast cost one shared-memory lookup per channel
// at most.  A hue op before contrast runs in both phases.
//
// Tiles as in gather.cu: a warp loads 512 pixels (1536 bytes) with three coalesced 16-byte loads per lane into a per-warp
// staging slice, then each lane converts 4 x 4 pixels and writes 512-byte float4 runs per plane.  T % 4 != 0 or an
// unaligned pointer takes the scalar loop of the same kernel (one pixel per thread, 4-byte stores).
#include "common.cuh"

namespace bpc {

constexpr int CJ_WARPS = 16;
constexpr int CJ_THREADS = CJ_WARPS * 32;
constexpr int CJ_TILE_PIX = 512;
constexpr int CJ_TILE_BYTES = CJ_TILE_PIX * 3;

enum { CJ_BRIGHTNESS = 0, CJ_CONTRAST = 1, CJ_SATURATION = 2, CJ_HUE = 3, CJ_TABLE = 4, CJ_NONE = -1 };

// A chain of at most four steps: CJ_TABLE (byte table), CJ_SATURATION (factor alpha), CJ_HUE or CJ_NONE.
struct CjProgram {
    int kind[4];
    float alpha[4];
    uint8_t tab[4][256];
};

struct CjShared {
    float lut[768];               // the caller's LUT (phase 2 reads olut)
    float olut[768];              // lut composed with the chain's trailing table run
    CjProgram slot;               // the order slots as given (phase 1 runs its prefix); contrast's table once the mean is known
    CjProgram prog;               // phase 2: `slot` with adjacent tables composed and a trailing table folded into olut
    float hfrac[256];             // HSV -> RGB: float32(h*6/255 - i), fs = float32(s/255), sector i % 6, per byte
    float hfs[256];
    uint8_t hsec[256];
    int wsum[CJ_WARPS];
    int mean;
    int nprog;
    __align__(16) uint8_t stage[CJ_WARPS][CJ_TILE_BYTES];
};

// Image.blend for one channel value (ImagingBlend, float alpha).
__device__ __forceinline__ int blend_px(int a, int x, float alpha) {
    const float v = __fadd_rn((float)a, __fmul_rn(alpha, (float)(x - a)));
    if (alpha >= 0.f && alpha <= 1.f) return __float2int_rz(v);
    return v <= 0.f ? 0 : v >= 255.f ? 255 : __float2int_rz(v);
}

__device__ __forceinline__ int luma(int r, int g, int b) { return (r * 19595 + g * 38470 + b * 7471 + 0x8000) >> 16; }

// C round (half away from zero) of a non-negative product, CLIP8.
__device__ __forceinline__ int cround8(double x) { return min(max((int)round(x), 0), 255); }

// Pillow's rgb2hsv_row, the byte shift of torchvision's adjust_hue, Pillow's hsv2rgb.
__device__ __forceinline__ void hue_px(int& r, int& g, int& b, int shift, const CjShared& sm) {
    const int mx = max(r, max(g, b)), mn = min(r, min(g, b));
    if (mx == mn) return;                                   // h = s = 0, and s == 0 maps back to (v, v, v)
    const float cr = (float)(mx - mn);
    const float s = __fdiv_rn(cr, (float)mx);
    auto ratio = [&](int c) { return (double)__fdiv_rn((float)(mx - c), cr); };
    double h;
    if (r == mx) h = dsub(ratio(b), ratio(g));
    else if (g == mx) h = dsub(dadd(2.0, ratio(r)), ratio(b));
    else h = dsub(dadd(4.0, ratio(g)), ratio(r));
    // Pillow divides by 6.0; the product with the rounded reciprocal differs from the quotient in at most the last bit
    // of the double, and on every one of the 2^24 colours the byte below comes out the same (tests/test_color_jitter.py)
    double x = dadd(dmul((double)__double2float_rn(h), 1.0 / 6.0), 1.0);
    if (x >= 1.0) x = dsub(x, 1.0);                         // fmod(x, 1.0): x is in [5/6, 2), the subtraction is exact
    const int uh = min(__double2int_rz(dmul((double)__double2float_rn(x), 255.0)), 255);
    const int us = min(__double2int_rz(dmul((double)s, 255.0)), 255);
    if (us == 0) {
        r = g = b = mx;
        return;
    }
    const int hh = (uh + shift) & 255;
    const double v = (double)mx, fs = (double)sm.hfs[us], f = (double)sm.hfrac[hh];
    const int p = cround8(dmul(v, dsub(1.0, fs)));
    const int q = cround8(dmul(v, dsub(1.0, dmul(fs, f))));
    const int t = cround8(dmul(v, dsub(1.0, dmul(fs, dsub(1.0, f)))));
    switch (sm.hsec[hh]) {
        case 0: r = mx; g = t; b = p; break;
        case 1: r = q; g = mx; b = p; break;
        case 2: r = p; g = mx; b = t; break;
        case 3: r = p; g = q; b = mx; break;
        case 4: r = t; g = p; b = mx; break;
        default: r = mx; g = p; b = q; break;
    }
}

// Steps [0, hi) of `pr` on N pixels.  The steps are uniform over the CTA, so every branch here is uniform.
template <int N>
__device__ __forceinline__ void chain(int (&r)[N], int (&g)[N], int (&b)[N], const CjProgram& pr, int hi, int shift, const CjShared& sm) {
#pragma unroll 1
    for (int k = 0; k < hi; ++k) {
        const int kind = pr.kind[k];
        if (kind == CJ_TABLE) {
            const uint8_t* t = pr.tab[k];
#pragma unroll
            for (int j = 0; j < N; ++j) {
                r[j] = t[r[j]]; g[j] = t[g[j]]; b[j] = t[b[j]];
            }
        } else if (kind == CJ_SATURATION) {
            const float a = pr.alpha[k];
#pragma unroll
            for (int j = 0; j < N; ++j) {
                const int L = luma(r[j], g[j], b[j]);
                r[j] = blend_px(L, r[j], a); g[j] = blend_px(L, g[j], a); b[j] = blend_px(L, b[j], a);
            }
        } else if (kind == CJ_HUE) {
#pragma unroll
            for (int j = 0; j < N; ++j) hue_px(r[j], g[j], b[j], shift, sm);
        }
    }
}

// One pass over crop `src` (P pixels).  SUM: apply steps [0, hi) of sm.slot and return this thread's share of the L sum.
// Otherwise apply steps [0, hi) of sm.prog and write the planes of `dst` through sm.olut (output plane 0 = channel 2 with SWAP).
template <bool SUM, bool SWAP>
__device__ __forceinline__ int pass(const uint8_t* __restrict__ src, float* __restrict__ dst, int P, bool vec, int hi, int shift,
                                    CjShared& sm) {
    const CjProgram& pr = SUM ? sm.slot : sm.prog;
    const float* lut = sm.olut;
    int sum = 0;
    if (!vec) {
        for (int p = threadIdx.x; p < P; p += CJ_THREADS) {
            int r[1] = {src[3 * p]}, g[1] = {src[3 * p + 1]}, b[1] = {src[3 * p + 2]};
            chain<1>(r, g, b, pr, hi, shift, sm);
            if (SUM) {
                sum += luma(r[0], g[0], b[0]);
            } else {
                dst[p] = lut[SWAP ? b[0] : r[0]];
                dst[P + p] = lut[256 + g[0]];
                dst[2 * (size_t)P + p] = lut[512 + (SWAP ? r[0] : b[0])];
            }
        }
        return sum;
    }
    const int lane = lane_id(), warp = warp_id();
    const int tiles = (P + CJ_TILE_PIX - 1) / CJ_TILE_PIX;
    int tile = warp;
    if (tile >= tiles) return 0;
    uint8_t* mine = sm.stage[warp];
    auto load = [&](int t, uint4 (&v)[3]) {
        const int bytes = min(CJ_TILE_BYTES, (P - t * CJ_TILE_PIX) * 3);
        const uint8_t* s = src + (size_t)t * CJ_TILE_BYTES;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int off = (k * 32 + lane) * 16;
            v[k] = off < bytes ? __ldg(reinterpret_cast<const uint4*>(s + off)) : make_uint4(0, 0, 0, 0);
        }
    };
    uint4 v[3];
    load(tile, v);
    while (true) {
#pragma unroll
        for (int k = 0; k < 3; ++k) *reinterpret_cast<uint4*>(mine + (k * 32 + lane) * 16) = v[k];
        __syncwarp();
        const int next = tile + CJ_WARPS;
        const bool more = next < tiles;
        if (more) load(next, v);
        const int npix = min(CJ_TILE_PIX, P - tile * CJ_TILE_PIX);
#pragma unroll 1
        for (int k = 0; k < 4; ++k) {
            const int q = k * 128 + lane * 4;               // 4 consecutive pixels = 12 bytes = 3 words
            if (q >= npix) break;
            const uint32_t* w = reinterpret_cast<const uint32_t*>(mine + q * 3);
            const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
            int r[4] = {(int)(w0 & 255u), (int)(w0 >> 24), (int)((w1 >> 16) & 255u), (int)((w2 >> 8) & 255u)};
            int g[4] = {(int)((w0 >> 8) & 255u), (int)(w1 & 255u), (int)(w1 >> 24), (int)((w2 >> 16) & 255u)};
            int b[4] = {(int)((w0 >> 16) & 255u), (int)((w1 >> 8) & 255u), (int)(w2 & 255u), (int)(w2 >> 24)};
            chain<4>(r, g, b, pr, hi, shift, sm);
            if (SUM) {
#pragma unroll
                for (int j = 0; j < 4; ++j) sum += luma(r[j], g[j], b[j]);
            } else {
                float* d = dst + (size_t)tile * CJ_TILE_PIX + q;
                const int* a = SWAP ? b : r;
                const int* c = SWAP ? r : b;
                __stcs(reinterpret_cast<float4*>(d), make_float4(lut[a[0]], lut[a[1]], lut[a[2]], lut[a[3]]));
                __stcs(reinterpret_cast<float4*>(d + P),
                       make_float4(lut[256 + g[0]], lut[256 + g[1]], lut[256 + g[2]], lut[256 + g[3]]));
                __stcs(reinterpret_cast<float4*>(d + 2 * (size_t)P),
                       make_float4(lut[512 + c[0]], lut[512 + c[1]], lut[512 + c[2]], lut[512 + c[3]]));
            }
        }
        if (!more) break;
        __syncwarp();
        tile = next;
    }
    return sum;
}

template <bool SWAP>
__global__ void __launch_bounds__(CJ_THREADS, 2)
bpc_color_jitter_kernel(const uint8_t* __restrict__ in, int T, const int32_t* __restrict__ order, const float* __restrict__ factors,
                        const float* __restrict__ lut_g, float* __restrict__ out, bool vec) {
    __shared__ CjShared sm;
    const int crop = blockIdx.x, tid = threadIdx.x;
    const int P = T * T;
    const uint8_t* src = in + (size_t)crop * P * 3;
    float* dst = out + (size_t)crop * 3 * P;
    int op[4];
    float fac[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        op[k] = __ldg(order + 4 * crop + k);
        fac[k] = __ldg(factors + 4 * crop + k);
    }
    int hi = 0, cpos = -1, has_hue = 0;                     // hi: slots up to the last real op; cpos: first contrast slot
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (op[k] >= 0 && op[k] <= 3) hi = k + 1;
        if (op[k] == CJ_CONTRAST && cpos < 0) cpos = k;
        has_hue |= op[k] == CJ_HUE;
    }
    const float fhue = __ldg(factors + 4 * crop + CJ_HUE);
    const int shift = has_hue ? (__double2int_rz(dmul((double)fhue, 255.0)) & 255) : 0;   // np.int32(f * 255).astype(uint8)
    for (int e = tid; e < 768; e += CJ_THREADS) sm.lut[e] = lut_g[e];
    if (tid < 4) {
        const int o = op[tid] >= 0 && op[tid] <= 3 ? op[tid] : CJ_NONE;
        sm.slot.kind[tid] = (o == CJ_BRIGHTNESS || o == CJ_CONTRAST) ? CJ_TABLE : o;
        sm.slot.alpha[tid] = (o >= 0) ? fac[o] : 0.f;
    }
    if (tid < 256) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (op[k] == CJ_BRIGHTNESS) sm.slot.tab[k][tid] = (uint8_t)blend_px(0, tid, fac[CJ_BRIGHTNESS]);
        if (has_hue) {
            const double x = ddiv(dmul((double)tid, 6.0), 255.0);
            const double i = floor(x);
            sm.hsec[tid] = (uint8_t)((int)i % 6);
            sm.hfrac[tid] = __double2float_rn(dsub(x, i));
            sm.hfs[tid] = __double2float_rn(ddiv((double)tid, 255.0));
        }
    }
    __syncthreads();
    if (cpos >= 0) {
        int s = pass<true, SWAP>(src, dst, P, vec, cpos, shift, sm);
        s = __reduce_add_sync(0xffffffffu, s);
        if (lane_id() == 0) sm.wsum[warp_id()] = s;
        __syncthreads();
        if (tid == 0) {
            int total = 0;                                  // <= 255 * 1024^2: fits
            for (int w = 0; w < CJ_WARPS; ++w) total += sm.wsum[w];
            sm.mean = __double2int_rz(dadd(ddiv((double)total, (double)P), 0.5));
        }
        __syncthreads();
        const int mean = sm.mean;
        if (tid < 256) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (op[k] == CJ_CONTRAST) sm.slot.tab[k][tid] = (uint8_t)blend_px(mean, tid, fac[CJ_CONTRAST]);
        }
        __syncthreads();
    }
    // Phase 2's program: each run of adjacent table slots composed into one table (thread v follows byte value v through
    // the run), the run at the end of the chain folded into the output LUT.
    if (tid < 256) {
        int v = tid, n = 0;
        bool run = false;
        for (int k = 0; k < hi; ++k) {
            const int kind = sm.slot.kind[k];
            if (kind == CJ_NONE) continue;
            if (kind == CJ_TABLE) {
                v = sm.slot.tab[k][v];
                run = true;
                continue;
            }
            if (run) {
                sm.prog.tab[n][tid] = (uint8_t)v;
                if (tid == 0) sm.prog.kind[n] = CJ_TABLE;
                ++n;
                v = tid;
                run = false;
            }
            if (tid == 0) {
                sm.prog.kind[n] = kind;
                sm.prog.alpha[n] = sm.slot.alpha[k];
            }
            ++n;
        }
        for (int c = 0; c < 3; ++c) sm.olut[256 * c + tid] = sm.lut[256 * c + v];
        if (tid == 0) sm.nprog = n;
    }
    __syncthreads();
    pass<false, SWAP>(src, dst, P, vec, sm.nprog, shift, sm);
}

}  // namespace bpc

using namespace bpc;

extern "C" int bpc_color_jitter(const uint8_t* in, int n, int T, const int32_t* order, const float* factors, int swap_rb,
                                const float* lut, float* out, void* stream) {
    if (n < 0 || T < 1 || T > BPC_MAX_TARGET) return BPC_EINVAL;
    if (n == 0) return BPC_OK;
    if (!in || !order || !factors || !lut || !out) return BPC_EINVAL;
    const bool vec = T % 4 == 0 && ((uintptr_t)in & 15) == 0 && ((uintptr_t)out & 15) == 0;
    auto fn = swap_rb ? bpc_color_jitter_kernel<true> : bpc_color_jitter_kernel<false>;
    fn<<<n, CJ_THREADS, 0, (cudaStream_t)stream>>>(in, T, order, factors, lut, out, vec);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}
