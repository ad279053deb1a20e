// The warp-specialised crop kernel: one crop per CTA, a producer warp feeding consumer warps (= 32-column strips) through a ring of
// TMA-filled slots.  Classes 1 (area, <= 3 taps), 3 (fixed-point bilinear) and 4 (area, 4 .. 6 taps) and rejected boxes; see
// crop.cu for the path as a whole and DESIGN.md 3.2 for the measurements behind the design.
#include <mutex>
#include <type_traits>

#include "crop_common.cuh"

namespace bpc {

// ------------------------------------------------------------------------------------------------------
// CTA kernel: classes 1, 3 and 4, one crop per CTA, warp-specialised
// ------------------------------------------------------------------------------------------------------
// Warps 0 .. NS-1 (NS = T / 32 strips) are consumers: one lane per output column, source rows in order.  The LAST warp is a
// producer whose lane 0 walks the list of class-1 / class-3 crops (atomic counter) and, per crop, copies the crop's block of
// row descriptors into shared memory (one bulk copy) and then, per ring slot, issues ONE 2-D tensor copy of eight FULL-WIDTH
// source rows -- seven times fewer TMA operations than one box per strip, every source byte fetched once per crop, and the
// ~300-cycle scoreboard wait behind each TMA issue (measured: 13 % of the per-strip kernel's warp time) sits in a warp that has
// nothing else to do.  The producer runs ahead across crops (ring of four slots, two descriptor blocks), which also hides
// the per-crop set-up round trips.  Consumers meet on the slots' full / empty mbarriers, so the strips of one crop stay within
// four slots of each other: whole 896-byte output rows of a plane reach L2 close together, and the rows above / below the
// resized image are written as contiguous runs by all consumer threads.
//   class 1 (area, <= 3 taps): per SOURCE row a (ba, bb) record (see bpc_crop_prep_kernel); a row whose ba has the sign bit
//            set closes the open output row (LUT, three 128-byte stores) and opens the next with weight bb;
//   class 3 (fixed-point bilinear, the box grows): per OUTPUT row (b0, b1, second source row, first source row); an output row
//            is emitted as soon as the slot holding its second source row has landed -- its first row is the previous output
//            row's first or second row, whose horizontal pass is still in registers.
// ring slots and resident CTAs per SM: the T = 224 float instantiation (the benchmark's) runs 4 CTAs/SM (8 warps, 63 registers,
// three slots: 55 KB of shared memory), which buys classes 3 and 4 latency hiding (0.66 -> 0.70, 0.67 -> 0.69) and leaves class 1
// where it was; the run-time-T and T = 256 instantiations (up to 9 warps) keep four slots and 3 CTAs/SM
__host__ __device__ constexpr int cta_nslot(int TT) { return TT == 224 ? 3 : 4; }
constexpr int CTA_NMAPS = 25;                // box widths 64, 128, ... 1600 bytes (8-byte elements)
struct CtaMaps { CUtensorMap m[CTA_NMAPS]; };
// staged bytes per source row of a crop: misalignment of its first byte + 3 w + what the widest horizontal pass over-reads
// (class 1: three words from the aligned tap address; class 4: up to six taps padded to the warp maximum)
__host__ __device__ __forceinline__ int cta_pitch(int mis0, int w, int cls) { return ((mis0 + 3 * w + (cls == 4 ? 40 : 12) + 63) >> 6) << 6; }
__host__ __device__ __forceinline__ int cta_desc_bytes(int T) { return ydesc_stride(T) * 16; }
__host__ __device__ __forceinline__ int cta_smem_bytes(int T, int nslot) { return LUT_SMEM + nslot * CTA_ROWS * cta_pitch_max(T) + 2 * cta_desc_bytes(T) + 256; }

// Lockstep of a crop's strips (a named barrier over the consumer warps): the seven 128-byte pieces of an output row then reach
// L2 within a short window and are written back together -- DRAM sees whole rows instead of scattered lines (measured on
// stores alone: 5.7 -> 7.2 TB/s; on the 60-400 px mix 0.79 -> 0.83 of roofline).  Class 1 only, once per ring slot: a barrier every
// eight output rows made class 3 slower (0.64 -> 0.57: many idle strips, latency-bound) and class 4 is issue-bound.
#define CTA_LOCKSTEP() do { if (cls == 1) asm volatile("bar.sync 1, %0;" :: "r"(NS * 32) : "memory"); } while (0)
__device__ __forceinline__ void mbar_arrive(unsigned bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory"); }

template <bool OUT_U8, int TT, bool SWAP, bool BF16 = false>
__global__ void __launch_bounds__(TT == 224 ? 256 : 288, TT == 224 ? 4 : 3)
bpc_crop_cta_kernel(const uint8_t* __restrict__ images, int B, int H, int W, const RoiGeom* __restrict__ geom,
                    const float4* __restrict__ xdesc, const float4* __restrict__ ydesc, const int32_t* __restrict__ list1,
                    int32_t* __restrict__ counters, int Trt, uchar4 fill, int swap_rb, const float* __restrict__ lut_g,
                    float* __restrict__ outf, uint8_t* __restrict__ outb, const __grid_constant__ CtaMaps tm) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int CTA_NSLOT = cta_nslot(TT);
    float* lut = reinterpret_cast<float*>(smem);
    const int T = TT ? TT : Trt;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int NS = (T + 31) >> 5;                                   // consumer warps; warp NS is the producer
    const int pitch_max = cta_pitch_max(T);
    const int slot_bytes = CTA_ROWS * pitch_max;
    const int desc_bytes = cta_desc_bytes(T);
    const unsigned smem_s = (unsigned)__cvta_generic_to_shared(smem);
    const unsigned ring_s = smem_s + LUT_SMEM;
    const unsigned desc_s = ring_s + CTA_NSLOT * slot_bytes;       // [2][ystride] float4: the current and the next crop's row descriptors
    const unsigned misc_s = desc_s + 2 * desc_bytes;
    const unsigned full_s = misc_s, empty_s = misc_s + 8 * CTA_NSLOT, hfull_s = misc_s + 16 * CTA_NSLOT, hempty_s = hfull_s + 16;
    volatile int* hdr = reinterpret_cast<volatile int*>(smem + (misc_s - smem_s) + 16 * CTA_NSLOT + 32);       // [2] crop index
    if (tid == 0) {
        for (int i = 0; i < CTA_NSLOT; ++i) { mbar_init(full_s + 8 * i, 1); mbar_init(empty_s + 8 * i, NS); }
        for (int i = 0; i < 2; ++i) { mbar_init(hfull_s + 8 * i, 1); mbar_init(hempty_s + 8 * i, NS); }
        *reinterpret_cast<volatile unsigned*>(smem + 3 * LUT_STRIDE * 4) = smem_s - 4u * 0x4B000000u;              // see lut_addr()
    }
    if (!OUT_U8)
        for (int e = tid; e < 768; e += (int)blockDim.x) lut[(e >> 8) * LUT_STRIDE + (e & 255)] = lut_g[e];
    __syncthreads();
    Out<OUT_U8, BF16> out;
    out_init(out, outf, outb, lut, T, swap_rb, fill);
    if (!OUT_U8 && tid < 3) lut[tid * LUT_STRIDE + 256] = out.padf[tid];
    __syncthreads();
    const unsigned lut_m = *reinterpret_cast<volatile unsigned*>(smem + 3 * LUT_STRIDE * 4);
    const int ds = desc_stride(T), ystride = ydesc_stride(T);
    const unsigned long long rowstride = (unsigned long long)W * 3ull;
    const unsigned long long img_end = (unsigned long long)(uintptr_t)images + (unsigned long long)B * H * rowstride;
    const int n1 = counters[8];
    int32_t* work = counters + 12;

    if (wid == NS) {
        // ------------------------------------ producer ------------------------------------
        if (lane != 0) return;
        // a list ordered by source row (bpc_crop_order_kernel) reads each source line again a few crops later: keep the lines in
        // L2 while the output streams past (evict-last; on boxes that do not overlap, which share nothing, it measured slower)
        const bool keep_src = counters[9] != 0;
        unsigned long long src_policy;
        asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(src_policy));
        int idx = atomicAdd(work, 1);
        unsigned cg = 0;                                            // slots filled so far
        for (int hi = 0;; ++hi) {
            const int hb = hi & 1;
            if (hi >= 2) mbar_wait(hempty_s + 8 * hb, ((hi >> 1) - 1) & 1);
            if (idx >= n1) {
                hdr[hb] = -1;
                mbar_arrive(hfull_s + 8 * hb);
                break;
            }
            const int idx_next = atomicAdd(work, 1);                // round trip hidden behind this crop's copies
            const int roi = list1[idx];
            const RoiGeom* gp = geom + roi;
            const unsigned long long src = gp->src;
            const int w = gp->w, h = gp->cls == 0 ? 0 : gp->h;     // a rejected box (class 0) has no source rows: header only
            hdr[hb] = roi;
            // the part of the crop's row-descriptor block that will be read: per output row (class 3) or per source row, padded slot included
            const unsigned dbytes = gp->cls == 0 ? 0u : (unsigned)min(desc_bytes, gp->cls == 3 ? 16 * (gp->new_h + 1) : 8 * (((h + CTA_ROWS - 1) & ~(CTA_ROWS - 1)) + CTA_ROWS));
            mbar_expect_tx(hfull_s + 8 * hb, dbytes);
            if (dbytes) bulk_g2s(desc_s + hb * desc_bytes, (unsigned long long)(uintptr_t)(ydesc + (size_t)roi * ystride), dbytes, hfull_s + 8 * hb);
            const int mis0 = (int)(src & 15ull);
            const int pitch = cta_pitch(mis0, w, gp->cls);
            const unsigned long long off = (src & ~15ull) - (unsigned long long)(uintptr_t)images;
            const int row0 = (int)(off / rowstride);
            const int x8 = (int)((off - (unsigned long long)row0 * rowstride) >> 3);
            if (gp->cls == 0) {
                // nothing to stage
            } else if (pitch <= pitch_max) {
                // one 2-D tensor copy of eight full-width rows per slot (rows / columns beyond the pool are zero-filled)
                const CUtensorMap* map = &tm.m[(pitch >> 6) - 1];
                const int nchunks = (h + CTA_ROWS - 1) / CTA_ROWS;
                for (int c = 0; c < nchunks; ++c, ++cg) {
                    const unsigned j = cg % CTA_NSLOT;
                    if (cg >= CTA_NSLOT) mbar_wait(empty_s + 8 * j, ((cg / CTA_NSLOT) - 1) & 1);
                    mbar_expect_tx(full_s + 8 * j, (unsigned)(CTA_ROWS * pitch));
                    if (keep_src)
                        asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
                                     :: "r"(ring_s + j * slot_bytes), "l"(map), "r"(x8), "r"(row0 + c * CTA_ROWS), "r"(full_s + 8 * j), "l"(src_policy) : "memory");
                    else
                        asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                                     :: "r"(ring_s + j * slot_bytes), "l"(map), "r"(x8), "r"(row0 + c * CTA_ROWS), "r"(full_s + 8 * j) : "memory");
                }
            } else {
                // wide class-4 crops (rows of up to 5 T pixels): rps rows per slot, one 1-D bulk copy each, clipped to the pool
                const int rps = slot_bytes / pitch;
                const int nchunks = (h + rps - 1) / rps;
                const unsigned long long a0 = src & ~15ull;
                for (int c = 0; c < nchunks; ++c, ++cg) {
                    const unsigned j = cg % CTA_NSLOT;
                    if (cg >= CTA_NSLOT) mbar_wait(empty_s + 8 * j, ((cg / CTA_NSLOT) - 1) & 1);
                    unsigned total = 0;
                    for (int r = 0; r < rps; ++r) {
                        const unsigned long long a = a0 + (unsigned long long)(c * rps + r) * rowstride;
                        if (a < img_end) total += (unsigned)min((unsigned long long)pitch, (img_end - a) & ~15ull);
                    }
                    mbar_expect_tx(full_s + 8 * j, total);
                    for (int r = 0; r < rps; ++r) {
                        const unsigned long long a = a0 + (unsigned long long)(c * rps + r) * rowstride;
                        if (a < img_end) {
                            const unsigned nb = (unsigned)min((unsigned long long)pitch, (img_end - a) & ~15ull);
                            if (nb) bulk_g2s(ring_s + j * slot_bytes + (unsigned)(r * pitch), a, nb, full_s + 8 * j);
                        }
                    }
                }
            }
            idx = idx_next;
        }
        return;
    }

    // ------------------------------------ consumers: warp = strip ------------------------------------
    constexpr bool swap = SWAP;
    const size_t plane = (size_t)T * T;
    const float nz = __int_as_float((int)(0x80000000u | (unsigned)fill.w));     // -0.0f: fill.w is 0 at run time
    const u64 nz2 = pack2(nz, nz);
    const int nthc = NS * 32;
    const int x = wid * 32 + lane;
    unsigned cg = 0;
    for (int hi = 0;; ++hi) {
        const int hb = hi & 1;
        mbar_wait(hfull_s + 8 * hb, (hi >> 1) & 1);
        const int roi = hdr[hb];
        if (roi < 0) break;
        const RoiGeom* gp = geom + roi;
        const int cls = gp->cls;
        const int new_w = gp->new_w, new_h = gp->new_h, dx0 = gp->dx, dy0 = gp->dy, h = gp->h;
        const int mis0 = (int)(gp->src & 15ull);
        const int pitch = cta_pitch(mis0, gp->w, cls);
        const int rps = pitch <= pitch_max ? CTA_ROWS : slot_bytes / pitch;       // source rows per ring slot
        const int nchunks = (h + rps - 1) / rps;
        const unsigned dsc = desc_s + hb * desc_bytes;
        if (cls == 0) {                                             // rejected box: the whole canvas is fill (no slots were issued)
            out.pad_rows(roi, 0, T, tid, nthc);
            __syncwarp();
            if (lane == 0) mbar_arrive(hempty_s + 8 * hb);
            continue;
        }
        out.pad_rows(roi, 0, dy0, tid, nthc);                       // whole rows above / below: contiguous runs
        out.pad_rows(roi, dy0 + new_h, T, tid, nthc);
        const int xr = x - dx0;
        const bool active = xr >= 0 && xr < new_w;
        const bool touches = wid * 32 < dx0 + new_w && wid * 32 + 32 > dx0;
        const bool store_ok = (TT && TT % 32 == 0) || x < T;
        float* optr = outf + ((size_t)roi * 3 * T + dy0) * T + x;     // (plane 0, first image row, column x)
        unsigned short* optr16 = reinterpret_cast<unsigned short*>(outf) + (((size_t)roi * T + dy0) * T + x) * 3;   // BF16: pixel (row, x), channels-last
        const unsigned short padh0 = bf16_bits(out.padf[0]), padh1 = bf16_bits(out.padf[1]), padh2 = bf16_bits(out.padf[2]);
        if (!touches) {
            // a strip beside the resized image: the fill value, at the pace of the neighbours
            int ydone = 0;
            for (int c = 0; c < nchunks; ++c, ++cg) {
                const unsigned j = cg % CTA_NSLOT;
                CTA_LOCKSTEP(); mbar_wait(full_s + 8 * j, (cg / CTA_NSLOT) & 1);
                __syncwarp();
                if (lane == 0) mbar_arrive(empty_s + 8 * j);
                int ndone;
                if (cls != 3) {
                    const float ba = (lane < rps) ? lds_f32(dsc + 8u * (unsigned)(c * rps + lane)) : 0.f;
                    ndone = __popc(__ballot_sync(0xffffffffu, __float_as_int(ba) < 0));
                } else {
                    // output rows whose second source row lies in this slot (monotone in y)
                    const int last_row = c * CTA_ROWS + CTA_ROWS - 1;
                    ndone = 0;
                    for (int y0 = ydone; y0 < new_h; y0 += 32) {
                        const int yy = y0 + lane;
                        const bool ok = yy < new_h && __float_as_int(lds_f4(dsc + 16u * (unsigned)min(yy, new_h - 1)).z) <= last_row;
                        const int n = __popc(__ballot_sync(0xffffffffu, ok));
                        ndone += n;
                        if (n < 32) break;
                    }
                }
                for (int r = 0; r < ndone; ++r) {
                    if (store_ok) {
                        if (OUT_U8) out.pad(roi, dy0 + ydone + r, x);
                        else if (BF16) { optr16[0] = padh0; optr16[1] = padh1; optr16[2] = padh2; optr16 += 3 * T; }
                        else { optr[0] = out.padf[0]; optr[plane] = out.padf[1]; optr[2 * plane] = out.padf[2]; optr += T; }
                    }
                }
                ydone += ndone;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(hempty_s + 8 * hb);         // done with this crop's descriptor block
            continue;
        }
        const float4 xd = xdesc[(size_t)roi * ds + min(max(xr, 0), new_w - 1)];
        const int xs = __float_as_int(xd.w) & 0xffffff;
        const int colc = 3 * xs + mis0;
        const unsigned colc4 = (unsigned)(colc & ~3);
        const int shc = (colc & 3) * 8;
        if (cls == 1) {
            ColW cw;
            cw.set(xd.x, xd.y, xd.z);
            if (!active) {                               // beside the image: every row sums to 256 -> LUT entry 256 = fill
                cw.w[0] = cw.w[1] = cw.w[2] = 0.f;
                cw.c[0] = 256.f; cw.c[1] = cw.c[2] = 0.f;
            }
            u64 acc01 = 0ull;
            float acc2 = 0.f;
            unsigned roff = 0;                                // element offset of the open output row from optr
            int yout = 0;
            for (int c = 0; c < nchunks; ++c, ++cg) {
                const unsigned j = cg % CTA_NSLOT;
                CTA_LOCKSTEP(); mbar_wait(full_s + 8 * j, (cg / CTA_NSLOT) & 1);
                const unsigned rbase = ring_s + j * slot_bytes + colc4;
                const unsigned rec = dsc + 8u * CTA_ROWS * (unsigned)c;
#pragma unroll
                for (int half = 0; half < CTA_ROWS / 4; ++half) {
                    const float4 dA = lds_f4(rec + 32u * half), dB = lds_f4(rec + 32u * half + 16);
                    u64 h01[4];
                    float h2[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) h_area3(rbase + (unsigned)((4 * half + k) * pitch), shc, cw, h01[k], h2[k]);
                    if (half == CTA_ROWS / 4 - 1) {
                        __syncwarp();                           // every lane has read slot j
                        if (lane == 0) mbar_arrive(empty_s + 8 * j);
                    }
                    const float ba[4] = {dA.x, dA.z, dB.x, dB.z}, bb[4] = {dA.y, dA.w, dB.y, dB.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float wa = fabsf(ba[k]);
                        acc01 = fadd2(acc01, fprod2(pack2(wa, wa), h01[k], nz2));
                        acc2 = __fadd_rn(acc2, __fmul_rn(wa, h2[k]));
                        if (__float_as_int(ba[k]) < 0) {            // output row complete
                            float a0f, a1f;
                            unpack2(acc01, a0f, a1f);
                            if (OUT_U8) {
                                if (active) out.px(roi, dy0 + yout, x, round_u8(a0f), round_u8(a1f), round_u8(acc2));
                                else if (x < T) out.pad(roi, dy0 + yout, x);
                                ++yout;
                            } else {
                                const unsigned l0 = lut_addr(a0f, lut_m), l1 = lut_addr(a1f, lut_m), l2 = lut_addr(acc2, lut_m);
                                if (store_ok) {
                                    const float v0 = lds_f32(swap ? l2 : l0), v1 = lds_f32(l1 + 4 * LUT_STRIDE), v2 = lds_f32((swap ? l0 : l2) + 8 * LUT_STRIDE);
                                    if (BF16) {
                                        unsigned short* o = optr16 + roff;
                                        o[0] = bf16_bits(v0); o[1] = bf16_bits(v1); o[2] = bf16_bits(v2);
                                    } else {
                                        float* o = optr + roff;
                                        stg_out<0>(o, v0); stg_out<1>(o + plane, v1); stg_out<2>(o + 2 * plane, v2);
                                    }
                                }
                                roff += BF16 ? 3u * (unsigned)T : (unsigned)T;
                            }
                            acc01 = fprod2(pack2(bb[k], bb[k]), h01[k], nz2);
                            acc2 = __fmul_rn(bb[k], h2[k]);
                        }
                    }
                }
            }
        } else if (cls == 4) {
            // ---------------- class 4: area, 4 .. 6 taps per axis, source rows in order ----------------
            const int xn = __float_as_int(xd.w) >> 24;
            const int nt = warp_max_i32(xn);                      // uniform: taps evaluated per source row
            float w[6], cc[6];
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                w[k] = (k == 0) ? xd.x : ((k < xn - 1) ? xd.y : ((k == xn - 1) ? xd.z : 0.f));
                if (!active) w[k] = 0.f;
                cc[k] = __fmul_rn(w[k], -8388608.0f);
                if (!active && k == 0) cc[k] = 256.f;             // beside the image: every row sums to 256 -> LUT entry 256 = fill
                asm volatile("" : "+f"(cc[k]));
            }
            u64 acc01 = 0ull;
            float acc2 = 0.f;
            unsigned roff = 0;
            int yout = 0;
            auto vstep = [&](float ba, float bb, u64 h01, float h2) {
                const float wa = fabsf(ba);
                acc01 = fadd2(acc01, fprod2(pack2(wa, wa), h01, nz2));
                acc2 = __fadd_rn(acc2, __fmul_rn(wa, h2));
                if (__float_as_int(ba) < 0) {                       // output row complete
                    float a0f, a1f;
                    unpack2(acc01, a0f, a1f);
                    if (OUT_U8) {
                        if (active) out.px(roi, dy0 + yout, x, round_u8(a0f), round_u8(a1f), round_u8(acc2));
                        else if (x < T) out.pad(roi, dy0 + yout, x);
                        ++yout;
                    } else {
                        const unsigned l0 = lut_addr(a0f, lut_m), l1 = lut_addr(a1f, lut_m), l2 = lut_addr(acc2, lut_m);
                        if (store_ok) {
                            const float v0 = lds_f32(swap ? l2 : l0), v1 = lds_f32(l1 + 4 * LUT_STRIDE), v2 = lds_f32((swap ? l0 : l2) + 8 * LUT_STRIDE);
                            if (BF16) {
                                unsigned short* o = optr16 + roff;
                                o[0] = bf16_bits(v0); o[1] = bf16_bits(v1); o[2] = bf16_bits(v2);
                            } else {
                                float* o = optr + roff;
                                stg_out<0>(o, v0); stg_out<1>(o + plane, v1); stg_out<2>(o + 2 * plane, v2);
                            }
                        }
                        roff += BF16 ? 3u * (unsigned)T : (unsigned)T;
                    }
                    acc01 = fprod2(pack2(bb, bb), h01, nz2);
                    acc2 = __fmul_rn(bb, h2);
                }
            };
            auto strip = [&](auto nt_c) {
                constexpr int NT = decltype(nt_c)::value;
                for (int c = 0; c < nchunks; ++c, ++cg) {
                    const unsigned j = cg % CTA_NSLOT;
                    CTA_LOCKSTEP(); mbar_wait(full_s + 8 * j, (cg / CTA_NSLOT) & 1);
                    const unsigned rbase = ring_s + j * slot_bytes + colc4;
                    const unsigned rec = dsc + 8u * (unsigned)(c * rps);
                    int r = 0;
                    for (; r + 1 < rps; r += 2) {                   // two rows at a time: their loads and conversions interleave
                        const float4 d = make_float4(lds_f32(rec + 8u * r), lds_f32(rec + 8u * r + 4), lds_f32(rec + 8u * r + 8), lds_f32(rec + 8u * r + 12));
                        u64 ha01, hb01;
                        float ha2, hb2;
                        h_area_n<NT>(rbase + (unsigned)(r * pitch), shc, w, cc, ha01, ha2);
                        h_area_n<NT>(rbase + (unsigned)((r + 1) * pitch), shc, w, cc, hb01, hb2);
                        vstep(d.x, d.y, ha01, ha2);
                        vstep(d.z, d.w, hb01, hb2);
                    }
                    if (r < rps) {
                        const float ba = lds_f32(rec + 8u * r), bb = lds_f32(rec + 8u * r + 4);
                        u64 ha01;
                        float ha2;
                        h_area_n<NT>(rbase + (unsigned)(r * pitch), shc, w, cc, ha01, ha2);
                        vstep(ba, bb, ha01, ha2);
                    }
                    __syncwarp();                               // every lane has read slot j
                    if (lane == 0) mbar_arrive(empty_s + 8 * j);
                }
            };
            if (nt <= 4) strip(std::integral_constant<int, 4>{});
            else if (nt == 5) strip(std::integral_constant<int, 5>{});
            else strip(std::integral_constant<int, 6>{});
        } else {
            // ---------------- class 3: fixed-point bilinear ----------------
            const int xw0 = __float_as_int(xd.x), xw1 = __float_as_int(xd.y);
            const unsigned lut_s = smem_s;
            int rowA = -1, rowB = -1;
            int HA[3] = {0, 0, 0}, HB[3] = {0, 0, 0};
            int y = 0;
            float4 d = lds_f4(dsc);
            for (int c = 0; c < nchunks; ++c, ++cg) {
                const unsigned j = cg % CTA_NSLOT;
                CTA_LOCKSTEP(); mbar_wait(full_s + 8 * j, (cg / CTA_NSLOT) & 1);
                const int last_row = c * CTA_ROWS + CTA_ROWS - 1;
                const unsigned sbase = ring_s + j * slot_bytes + colc4 - (unsigned)(c * CTA_ROWS * pitch);     // source row r at sbase + r * pitch
                while (y < new_h) {
                    // (b * H) >> 16 as the high word of (b << 16) * H: one IMAD.HI instead of a multiply and a shift (0 <= b <= 2048, 0 <= H < 2^15)
                    const unsigned b0 = (unsigned)__float_as_int(d.x) << 16, b1 = (unsigned)__float_as_int(d.y) << 16;
                    const int sy0 = __float_as_int(d.w), sy1 = __float_as_int(d.z);
                    if (sy1 > last_row) break;
                    ++y;
                    d = lds_f4(dsc + 16u * (unsigned)y);              // next row's descriptor behind this row's arithmetic
                    if (active) {
                        if (sy0 != rowA) {
                            if (sy0 == rowB) { HA[0] = HB[0]; HA[1] = HB[1]; HA[2] = HB[2]; }
                            else h_lin(sbase + (unsigned)(sy0 * pitch), shc, xw0, xw1, HA);
                            rowA = sy0;
                        }
                        if (sy1 != rowB) {
                            if (sy1 == rowA) { HB[0] = HA[0]; HB[1] = HA[1]; HB[2] = HA[2]; }
                            else h_lin(sbase + (unsigned)(sy1 * pitch), shc, xw0, xw1, HB);
                            rowB = sy1;
                        }
                        unsigned o[3];                      // 4 * value + 2 low bits
#pragma unroll
                        for (int k = 0; k < 3; ++k) o[k] = __umulhi(b1, (unsigned)HB[k]) + (__umulhi(b0, (unsigned)HA[k]) + 2u);
                        if (OUT_U8) {
                            out.px(roi, dy0 + y - 1, x, (int)(o[0] >> 2) & 255, (int)(o[1] >> 2) & 255, (int)(o[2] >> 2) & 255);
                        } else {
                            const float v0 = lds_f32(lut_s + ((swap ? o[2] : o[0]) & 0x3fcu)), v1 = lds_f32(lut_s + 4 * LUT_STRIDE + (o[1] & 0x3fcu)),
                                        v2 = lds_f32(lut_s + 8 * LUT_STRIDE + ((swap ? o[0] : o[2]) & 0x3fcu));
                            if (BF16) {
                                optr16[0] = bf16_bits(v0); optr16[1] = bf16_bits(v1); optr16[2] = bf16_bits(v2);
                                optr16 += 3 * T;
                            } else {
                                stg_out<0>(optr, v0); stg_out<1>(optr + plane, v1); stg_out<2>(optr + 2 * plane, v2);
                                optr += T;
                            }
                        }
                    } else if (x < T) {
                        if (OUT_U8) out.pad(roi, dy0 + y - 1, x);
                        else if (BF16) { optr16[0] = padh0; optr16[1] = padh1; optr16[2] = padh2; optr16 += 3 * T; }
                        else { optr[0] = out.padf[0]; optr[plane] = out.padf[1]; optr[2 * plane] = out.padf[2]; optr += T; }
                    }
                }
                __syncwarp();                               // every lane is done with slot j
                if (lane == 0) mbar_arrive(empty_s + 8 * j);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(hempty_s + 8 * hb);             // done with this crop's descriptor block
    }
}

// Tensor maps of the CTA kernel: the pool as [B*H rows][W*3/8 uint64], box = {64 i bytes, CTA_ROWS rows}, i = 1 .. CTA_NMAPS.
static int cta_tensor_maps(const uint8_t* images, int B, int H, int W, CtaMaps* out) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static std::mutex mu;
    static CtaMaps cached;
    static const uint8_t* k_images = nullptr;
    static int k_B = 0, k_H = 0, k_W = 0, k_dev = -1;
    static EncodeFn encode = nullptr;
    std::lock_guard<std::mutex> lock(mu);
    int dev = 0;
    cudaGetDevice(&dev);
    if (images == k_images && B == k_B && H == k_H && W == k_W && dev == k_dev) { *out = cached; return BPC_OK; }
    if (!encode) {
        cudaDriverEntryPointQueryResult q;
        void* fnp = nullptr;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fnp, cudaEnableDefault, &q);
        if (e != cudaSuccess) return (int)e;
        if (q != cudaDriverEntryPointSuccess || !fnp) return (int)cudaErrorNotSupported;
        encode = (EncodeFn)fnp;
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)W * 3 / 8, (cuuint64_t)B * H};
    const cuuint64_t gstride[1] = {(cuuint64_t)W * 3};
    const cuuint32_t estr[2] = {1, 1};
    for (int i = 0; i < CTA_NMAPS; ++i) {
        const cuuint32_t box[2] = {(cuuint32_t)(8 * (i + 1)), (cuuint32_t)CTA_ROWS};
        const CUresult r = encode(&cached.m[i], CU_TENSOR_MAP_DATA_TYPE_UINT64, 2, (void*)images, gdim, gstride, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, BPC_L2_PROMO,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { k_images = nullptr; return (int)cudaErrorInvalidValue; }
    }
    k_images = images; k_B = B; k_H = H; k_W = W; k_dev = dev;
    *out = cached;
    return BPC_OK;
}

int crop_cta_launch(int out_mode, const uint8_t* images, int B, int H, int W, const RoiGeom* geom, const float4* xdesc, const float4* ydesc,
                    const int32_t* list1, int32_t* counters, int R, int T, uchar4 fill, int swap_rb, const float* lut, float* outf,
                    uint8_t* outb, cudaStream_t st) {
    typedef void (*CtaFn)(const uint8_t*, int, int, int, const RoiGeom*, const float4*, const float4*, const int32_t*, int32_t*, int,
                          uchar4, int, const float*, float*, uint8_t*, const CtaMaps);
    CtaMaps cmaps;
    const int terr = cta_tensor_maps(images, B, H, W, &cmaps);
    if (terr != BPC_OK) return terr;
    const bool sw = swap_rb != 0;
    CtaFn fn;
    if (out_mode == 1) fn = bpc_crop_cta_kernel<true, 0, false>;
    else if (out_mode == 2) fn = sw ? bpc_crop_cta_kernel<false, 0, true, true> : bpc_crop_cta_kernel<false, 0, false, true>;
    else if (T == 224) fn = sw ? bpc_crop_cta_kernel<false, 224, true> : bpc_crop_cta_kernel<false, 224, false>;
    else if (T == 256) fn = sw ? bpc_crop_cta_kernel<false, 256, true> : bpc_crop_cta_kernel<false, 256, false>;
    else fn = sw ? bpc_crop_cta_kernel<false, 0, true> : bpc_crop_cta_kernel<false, 0, false>;
    const int nslot = cta_nslot((out_mode == 0 && T == 224) ? 224 : 0);      // as the instantiation picked above
    const int smem_bytes = cta_smem_bytes(T, nslot);
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, cta_smem_bytes(T == 224 ? 224 : CTA_MAX_T, nslot));
    if (e != cudaSuccess) return (int)e;
    const int threads = 32 * ((T + 31) / 32 + 1);
    int dev = 0, sms = 148, per_sm = 3;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, smem_bytes) != cudaSuccess || per_sm < 1) per_sm = 1;
    const long long slots = (long long)sms * per_sm;
    const int grid = (int)((long long)R < slots ? R : slots);
    fn<<<grid, threads, smem_bytes, st>>>(images, B, H, W, geom, xdesc, ydesc, list1, counters, T, fill, swap_rb, lut, outf, outb, cmaps);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

}  // namespace bpc
