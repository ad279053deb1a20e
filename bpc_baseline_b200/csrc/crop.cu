// ROI crop -> aspect-preserving letterbox (cv2.resize INTER_AREA) -> colour order -> normalise.
//
// Replaces letterbox_preserving_aspect_ratio (bpc/utils/data_utils.py:34-44) and the inline transform
// of PoseEstimator._estimate_rotation (bpc/inference/process_pose.py:199-209).  The uint8 resize is
// bit-exact with OpenCV's INTER_AREA for 8UC3 (SURVEY.md App. C):
//   regime 1  both axes shrink           : float32 area taps, sequential mul/add (no FMA), cvRound
//   regime 2  both shrink, integer ratio : integer box sum; 2x2 -> (sum+2)>>2
//   regime 3  either axis grows          : 11-bit fixed-point bilinear with area-mode coordinates
//
// Kernels of one call (shared pieces in crop_common.cuh):
//   bpc_crop_prep     one CTA per ROI: letterbox geometry (float64, as Python / OpenCV compute it), regime
//                     and class of the ROI, and -- for the fast classes -- the per-column and per-row tap
//                     descriptors (start index + float32 weights, absent taps = +0.0f; per-SOURCE-row records for
//                     the area classes), so that no float64 arithmetic is left in the hot kernels; sorts the ROIs
//                     into the lists of the kernels below;
//   bpc_crop_cta      (crop_cta.cu) THE hot kernel: one crop per CTA, a producer warp issuing one full-width 2-D TMA
//                     box of eight source rows per ring slot, consumer warps = 32-column strips.  Classes 1 (regime
//                     1, scale < 2, <= 3 taps per axis; scale exactly 1), 3 (regime 3) and 4 (regime 1 with 4..6 taps
//                     per axis, 2 <= scale <= 5) and rejected boxes, whenever the image pitch is a multiple of 16
//                     bytes, at least WARP_MAX_PITCH and cta_pitch_max(T), and T <= 256;
//   bpc_crop_warp     the same classes on every other pool (other pitches, narrow images, T > 256): persistent CTAs,
//                     the unit of work is (ROI, strip of 32 output columns), taken by ONE WARP from a global atomic
//                     counter, plus one "padding" item per ROI; each warp stages its strip's source rows with one
//                     1-D bulk copy per row (guarded cp.async for the last bytes of the pool);
//   bpc_crop_generic  persistent CTAs over the (rare) remaining ROIs (class 2): integer ratios >= 2, scale > 5,
//                     source rows streamed through shared memory in chunks (boxes as large as the image).
// The dominant traffic is the float32 output (3*T*T*4 B per ROI): each warp stores 128 contiguous bytes per
// plane and row; padding rows are written with 16-byte stores.
#include <cooperative_groups.h>

#include <type_traits>

#include "crop_common.cuh"

namespace bpc {

#ifndef BPC_PREP_THREADS
#define BPC_PREP_THREADS 128
#endif
constexpr int PREP_THREADS = BPC_PREP_THREADS;      // threads of a prep CTA (one ROI each); 128: twice the CTAs in flight of 256 behind the serial geometry section (-33 us per 16 384 ROIs)

// Per-SOURCE-row records of an area resize with at most `maxtaps` taps per output row (collective over the PREP_THREADS threads of a prep
// CTA): record s = (ba, bb); |ba| = weight of source row s in the output row being accumulated, sign bit of ba set = that output
// row is complete after row s; bb = weight of row s as the first tap of the next output row (+0 if it has none there).  Rows
// [h, hpad) stay zero (no contribution, no completed row) so that whole ring slots run to completion.  *bad is set when the taps
// do not have this shape (then the ROI takes the generic path).
__device__ void src_row_records(float2* ysrc, int cap, const RoiGeom& g, int maxtaps, int tid, int* bad) {
    const int hpad = min(cap, ((g.h + CTA_ROWS - 1) / CTA_ROWS) * CTA_ROWS + CTA_ROWS);
    if (g.h + CTA_ROWS > cap) *bad = 1;
    for (int s = tid; s < hpad; s += PREP_THREADS) ysrc[s] = make_float2(0.f, 0.f);
    __syncthreads();
    for (int d = tid; d < g.new_h && !*bad; d += PREP_THREADS) {
        int ys, yn, fl; float bf, bm, bl;
        area_taps(d, g.scale_y, g.h, ys, yn, bf, bm, bl, fl);
        const int prev_last = d > 0 ? area_last_tap(d - 1, g.scale_y, g.h) : -1;
        if (yn < 1 || yn > maxtaps || ys < prev_last || ys + yn > g.h) { *bad = 1; break; }
        for (int t = 0; t < yn; ++t) {
            const int s = ys + t;
            const bool shared_first = (t == 0 && s == prev_last);       // row s also closes output row d - 1
            if (shared_first && yn == 1) { *bad = 1; break; }           // one source row closing two output rows: generic path
            float wv = (t == 0 && (fl & 1)) ? bf : ((t == yn - 1 && (fl & 2)) ? bl : bm);
            if (t == yn - 1) wv = __int_as_float(__float_as_int(wv) | (int)0x80000000u);
            if (shared_first) ysrc[s].y = wv; else ysrc[s].x = wv;
        }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------------
// prep: geometry, classification and tap descriptors, one CTA per ROI
// ------------------------------------------------------------------------------------------------------
// Descriptor formats (float4; desc_stride(T) per ROI on the x axis, desc_stride(T) + 8 on the y axis):
//   class 1 (area, <= 3 taps)  x: (w0, w1, w2, bits(first source column))
//                              y: (b0, b1, b2, bits(first source row | taps << 24))          [warp kernel]
//                              y: float2 per SOURCE row s [CTA kernel]: (ba, bb).  |ba| = weight of row s in the
//                                 output row being accumulated; sign bit of ba set = that output row is complete after row s;
//                                 bb = weight of row s as the first tap of the next output row (+0 if it has none there).
//                                 An output row then is acc = (((0 + b0 h0) + b1 h1) + b2 h2), bit-identical to OpenCV's
//                                 sum = b0 h0; sum += b1 h1; ... for non-negative terms.
//   class 3 (fixed-point)      x: (bits(w0), bits(w1), 0, bits(source column))      w = 2048, 0 beyond xmax
//                              y: (bits(b0), bits(b1), bits(second source row), bits(first source row))
// Ten CTAs per SM (48 registers): left to itself ptxas 12.9 picks 50, which allocates as 56 and leaves room for nine
__global__ void __launch_bounds__(PREP_THREADS, 10)
bpc_crop_prep_kernel(const uint8_t* __restrict__ images, int B, int H, int W, const int32_t* __restrict__ rois,
                     const int32_t* __restrict__ n_rois_dev, int roi_first, int T, int use_cta,
                     RoiGeom* __restrict__ geom, float4* __restrict__ xdesc, float4* __restrict__ ydesc,
                     int32_t* __restrict__ glist, int32_t* __restrict__ gcount, int32_t* __restrict__ status, int32_t* __restrict__ list1) {
    __shared__ RoiGeom g;
    __shared__ int s_bad;
    const int roi = blockIdx.x, tid = threadIdx.x;
    const int ds = desc_stride(T);
    if (tid == 0) {
        s_bad = 0;
        g.scale_x = g.scale_y = g.inv_x = g.inv_y = 0.0;
        g.src = 0ull;
        g.new_w = g.new_h = g.dx = g.dy = 0;
        g.regime = 0; g.cls = 0; g.isx = g.isy = 0; g.pitch = 16; g.pad_ = 0;
        const int32_t* r = rois + (size_t)roi * 5;
        const int img = r[0], x1 = r[1], y1 = r[2], x2 = r[3], y2 = r[4];
        const int w = x2 - x1, h = y2 - y1;
        g.w = w; g.h = h;
        if (n_rois_dev != nullptr && roi_first + roi >= *n_rois_dev) {
            g.cls = -1;
        } else {
            if (img >= 0 && img < B && x1 >= 0 && y1 >= 0 && x2 <= W && y2 <= H && w > 0 && h > 0 && w <= BPC_MAX_ROI_WIDTH) {
                // letterbox geometry, data_utils.py:35-38,41-42 (Python round = half-to-even on the f64 product)
                const double scale = ddiv((double)T, (double)max(h, w));
                const int new_w = (int)__double2ll_rn(dmul((double)w, scale));
                const int new_h = (int)__double2ll_rn(dmul((double)h, scale));
                if (new_w >= 1 && new_h >= 1 && new_w <= T && new_h <= T) {
                    g.new_w = new_w; g.new_h = new_h;
                    g.dx = (T - new_w) / 2; g.dy = (T - new_h) / 2;
                    g.inv_x = ddiv((double)new_w, (double)w);      // cv2.resize: inv_scale = dsize / ssize
                    g.inv_y = ddiv((double)new_h, (double)h);
                    g.scale_x = ddiv(1.0, g.inv_x);
                    g.scale_y = ddiv(1.0, g.inv_y);
                    if (g.scale_x >= 1.0 && g.scale_y >= 1.0) {
                        g.isx = __double2int_rn(g.scale_x);
                        g.isy = __double2int_rn(g.scale_y);
                        const bool fast = fabs(dsub(g.scale_x, (double)g.isx)) < 2.220446049250313e-16 &&
                                          fabs(dsub(g.scale_y, (double)g.isy)) < 2.220446049250313e-16;
                        g.regime = fast ? 2 : 1;
                    } else {
                        g.regime = 3;
                    }
                    g.src = (unsigned long long)(uintptr_t)images + (((unsigned long long)img * H + y1) * W + x1) * 3ull;
                    // scale exactly 1 (long side == T) is OpenCV's integer-ratio regime, but a 1 x 1 box sum is the byte itself and
                    // so is the area pass with its single tap of weight 1.0f: keep it on the fast path
                    if ((g.regime == 1 && g.scale_x < 2.0 && g.scale_y < 2.0) || (g.regime == 2 && g.isx == 1 && g.isy == 1)) g.cls = 1;
                    else if (g.regime == 3) g.cls = 3;
                    else if (g.regime == 1) {
                        // general tap counts in the warp kernel if a strip's rows fit its staging buffer:
                        // 32 columns span at most 31*scale_x + ceil(scale_x) + 2 source pixels
                        const int seg_px = (int)(31.0 * g.scale_x) + (int)ceil(g.scale_x) + 3;
                        const int pitch_max = ((3 * seg_px + 46) >> 4) << 4;
                        const bool taps6 = (int)ceil(g.scale_x) + 1 <= 6 && (int)ceil(g.scale_y) + 1 <= 6;
                        // warp kernel: a strip's rows fit its staging ring; CTA kernel (full-width rows): any width
                        g.cls = (taps6 && (use_cta || pitch_max <= WARP_MAX_PITCH)) ? 4 : 2;
                    } else g.cls = 2;
                }
            }
            if (status != nullptr) status[roi] = (g.regime == 0) ? 1 : 0;
        }
    }
    __syncthreads();
    const int cls = g.cls;
    float4* xd = xdesc + (size_t)roi * ds;
    float4* yd = ydesc + (size_t)roi * ydesc_stride(T);
    if (cls == 4) {
        // (w_first, w_middle, w_last, bits(start | taps << 24)); a missing first / last tap takes the middle weight
        for (int axis = 0; axis < (use_cta ? 1 : 2); ++axis) {
            const int nd = axis ? g.new_h : g.new_w;
            for (int d = tid; d < nd; d += PREP_THREADS) {
                int st, n, flags; float af, am, al;
                area_taps(d, axis ? g.scale_y : g.scale_x, axis ? g.h : g.w, st, n, af, am, al, flags);
                const float w0 = (flags & 1) ? af : ((n == 1 && (flags & 2)) ? al : am);
                const float wl = (flags & 2) ? al : am;
                (axis ? yd : xd)[d] = make_float4(w0, am, wl, __int_as_float(st | (n << 24)));
            }
        }
        if (use_cta) {
            src_row_records(reinterpret_cast<float2*>(yd), 2 * ydesc_stride(T), g, 6, tid, &s_bad);
            if (s_bad && tid == 0) { g.cls = 2; }
        }
    } else if (cls == 1) {
        for (int d = tid; d < g.new_w; d += PREP_THREADS) {
            int xs, xn; float w0, w1, w2;
            area_taps3(d, g.scale_x, g.w, xs, xn, w0, w1, w2);
            xd[d] = make_float4(w0, w1, w2, __int_as_float(xs));
        }
        if (use_cta) {
            src_row_records(reinterpret_cast<float2*>(yd), 2 * ds + YSRC_PAD, g, 3, tid, &s_bad);
            if (s_bad && tid == 0) { g.cls = 2; }
        } else {
            for (int d = tid; d < g.new_h; d += PREP_THREADS) {
                int ys, yn; float b0, b1, b2;
                area_taps3(d, g.scale_y, g.h, ys, yn, b0, b1, b2);
                yd[d] = make_float4(b0, b1, b2, __int_as_float(ys | (yn << 24)));
            }
        }
    } else if (cls == 3) {
        for (int d = tid; d < g.new_w; d += PREP_THREADS) {
            int xs, w0, w1, edge;
            linear_coef(d, g.scale_x, g.inv_x, g.w, xs, w0, w1, edge);
            if (edge) { w0 = 2048; w1 = 0; }                        // D = S[sx] * ONE beyond xmax
            xd[d] = make_float4(__int_as_float(w0), __int_as_float(w1), 0.f, __int_as_float(xs));
        }
        for (int d = tid; d < g.new_h; d += PREP_THREADS) {
            int s0, b0, b1, edge;
            linear_coef(d, g.scale_y, g.inv_y, g.h, s0, b0, b1, edge);
            const int s1 = min(s0 + 1, g.h - 1);
            yd[d] = make_float4(__int_as_float(b0), __int_as_float(b1), __int_as_float(s1), __int_as_float(s0));
        }
    }
    __syncthreads();
    if (tid == 0) {
        if (g.cls == 2) glist[atomicAdd(gcount, 1)] = roi;
        else if (use_cta && g.cls != -1) list1[atomicAdd(gcount + 8, 1)] = roi;     // classes 0, 1, 3, 4: the CTA kernel's list
        geom[roi] = g;
    }
}

// ------------------------------------------------------------------------------------------------------
// order of the CTA kernel's list: crops by their first source row in the pool
// ------------------------------------------------------------------------------------------------------
// The prep kernel appends the list in about ROI order, which for a batch of scenes is scene order: when scenes share
// captures (a pool of images) or their detections overlap, a source line is needed again only hundreds of crops later,
// after more output than the 126 MB L2 holds has streamed through it.  Sorted by first source row (image * H + y1), the
// crops in flight read a narrow band of the pool and the repeated lines come from L2.  Outputs do not change: each crop
// writes its own slot only, the order decides when it runs.
// Only a list whose crops read more source pixels than the pool holds is reordered: every pool pixel is then read more
// than once on average, so the crops must share lines.  Where they share less (boxes that do not overlap, small boxes in
// a large pool) the new order buys nothing and scatters the output slots being written (3-4 % slower, DESIGN.md 3.2),
// and the list stays as prep wrote it.  counters[9] = 1 marks a reordered list (the CTA kernel then keeps the source
// lines in L2 with an evict-last policy).
// One cluster of ORDER_CTAS CTAs, each over a slice of the list (one CTA over the whole list took 40 us per 16 384 entries,
// the cluster 15 us; DESIGN.md 3.2): per CTA a shared-memory histogram over buckets of
// 2^shift rows (shift the least that leaves at most ORDER_BUCKETS of them in [0, B H)); through distributed shared memory
// every CTA adds up the cluster's counts per bucket and those of the lower-ranked CTAs, scans them and scatters its entries
// into the unused tail of the generic list (glist[gcount, R) holds at least n1 entries, as gcount + n1 <= R); after a
// cluster barrier each CTA copies its slice back into list1.  Ties (crops in one bucket) fall in any order.
constexpr int ORDER_CTAS = 8;
constexpr int ORDER_THREADS = 1024;
constexpr int ORDER_BUCKETS = 4096;
constexpr int ORDER_BATCH = 6;                // list entries per thread with their loads in flight together

__global__ void __cluster_dims__(ORDER_CTAS, 1, 1) __launch_bounds__(ORDER_THREADS)
bpc_crop_order_kernel(const uint8_t* __restrict__ images, int B, int H, int W, const RoiGeom* __restrict__ geom,
                      int32_t* __restrict__ list1, int32_t* __restrict__ counters, int32_t* __restrict__ glist) {
    namespace cg = cooperative_groups;
    __shared__ __align__(16) int cnt[ORDER_BUCKETS];   // this CTA's entries per bucket (read by the whole cluster)
    __shared__ int pos[ORDER_BUCKETS];            // next list slot of this CTA's entries per bucket
    __shared__ int wsum[ORDER_THREADS / 32];
    __shared__ unsigned long long wpx[ORDER_THREADS / 32], s_px;
    const int n = counters[8];
    if (n < 2) return;
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int per = (n + ORDER_CTAS - 1) / ORDER_CTAS;
    const int lo = min(n, rank * per), hi = min(n, lo + per);
    int32_t* tmp = glist + counters[0];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned long long base = (unsigned long long)(uintptr_t)images, rowstride = (unsigned long long)W * 3ull;
    const unsigned long long rows = (unsigned long long)B * H;
    const double inv_rowstride = 1.0 / (double)rowstride;
    const int shift = max(0, 64 - __clzll((long long)rows - 1) - 12);          // (B H - 1) >> shift < ORDER_BUCKETS
    for (int b = tid; b < ORDER_BUCKETS; b += ORDER_THREADS) cnt[b] = 0;
    __syncthreads();
    // visit(roi, bucket, w h) for the entries [lo, hi) (w h = 0 unless `area`).  First source row = (src - images) / (3 W):
    // the double quotient is within one row of the exact one (no 64-bit division).  A rejected box (class 0, src = 0) has
    // no source rows and goes to bucket 0.
    auto pass = [&](bool area, auto&& visit) {
        for (int i0 = lo; i0 < hi; i0 += ORDER_THREADS * ORDER_BATCH) {
            int roi[ORDER_BATCH];
            unsigned long long src[ORDER_BATCH];
            int2 wh[ORDER_BATCH];
#pragma unroll
            for (int k = 0; k < ORDER_BATCH; ++k) {
                const int i = i0 + k * ORDER_THREADS + tid;
                roi[k] = i < hi ? list1[i] : -1;
            }
#pragma unroll
            for (int k = 0; k < ORDER_BATCH; ++k) {
                src[k] = roi[k] >= 0 ? geom[roi[k]].src : 0ull;
                wh[k] = roi[k] >= 0 && area ? *reinterpret_cast<const int2*>(&geom[roi[k]].w) : make_int2(0, 0);
            }
#pragma unroll
            for (int k = 0; k < ORDER_BATCH; ++k) {
                if (roi[k] < 0) continue;
                int b = 0;
                if (src[k]) {
                    const unsigned long long off = src[k] - base;
                    unsigned long long row = (unsigned long long)((double)off * inv_rowstride);
                    if (row * rowstride > off) --row;
                    else if ((row + 1) * rowstride <= off) ++row;
                    b = (int)(row >> shift);
                }
                visit(roi[k], b, src[k] ? (unsigned long long)wh[k].x * (unsigned long long)wh[k].y : 0ull);
            }
        }
    };
    unsigned long long px = 0ull;                                   // source pixels of this thread's crops
    pass(true, [&](int, int b, unsigned long long a) { atomicAdd(&cnt[b], 1); px += a; });
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) px += __shfl_down_sync(0xffffffffu, px, d);
    if (lane == 0) wpx[wid] = px;
    __syncthreads();
    if (tid == 0) {
        unsigned long long t = 0ull;
        for (int w = 0; w < ORDER_THREADS / 32; ++w) t += wpx[w];
        s_px = t;
    }
    cluster.sync();                                                 // every CTA's counts and pixel sum are complete
    unsigned long long list_px = 0ull;
    for (int r = 0; r < ORDER_CTAS; ++r) list_px += *cluster.map_shared_rank(&s_px, r);
    if (list_px <= rows * (unsigned long long)W) {                  // the same decision in every CTA
        cluster.sync();                                             // no CTA reads another's shared memory after this
        return;
    }
    constexpr int PER = ORDER_BUCKETS / ORDER_THREADS;
    static_assert(PER * ORDER_THREADS == ORDER_BUCKETS && ORDER_THREADS == 1024, "four buckets per thread, 32 warps");
    int c[PER], below[PER], s = 0;
#pragma unroll
    for (int k = 0; k < PER; ++k) c[k] = below[k] = 0;
    for (int r = 0; r < ORDER_CTAS; ++r) {                          // one 16-byte remote load per rank and thread
        const int4 v = reinterpret_cast<const int4*>(cluster.map_shared_rank(cnt, r))[tid];
        const int vk[PER] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            c[k] += vk[k];
            if (r < rank) below[k] += vk[k];
        }
    }
    cluster.sync();                                                 // no CTA reads another's shared memory after this
#pragma unroll
    for (int k = 0; k < PER; ++k) s += c[k];
    int incl = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) wsum[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        const int v = wsum[lane];
        int iv = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, iv, d);
            if (lane >= d) iv += u;
        }
        wsum[lane] = iv - v;
    }
    __syncthreads();
    int run = wsum[wid] + incl - s;
#pragma unroll
    for (int k = 0; k < PER; ++k) { pos[tid * PER + k] = run + below[k]; run += c[k]; }
    __syncthreads();
    pass(false, [&](int roi, int b, unsigned long long) { tmp[atomicAdd(&pos[b], 1)] = roi; });
    cluster.sync();                                                 // the whole list is in tmp (release / acquire over the cluster)
    for (int i = lo + tid; i < hi; i += ORDER_THREADS) list1[i] = tmp[i];
    if (rank == 0 && tid == 0) counters[9] = 1;
}

// ------------------------------------------------------------------------------------------------------
// warp kernel: (ROI, 32-column strip) items, one warp each
// ------------------------------------------------------------------------------------------------------
// Stage rows [s_lo, s_lo + count) of a strip into a warp buffer.  Normal case: one TMA bulk copy of `pitch` bytes
// per row (lane r issues row r), completion counted in bytes on the warp's mbarrier -> returns 1.  If the
// 16-byte-aligned over-read of the last row would leave the image pool (last rows of the last image) the
// rows are copied with guarded 16-byte cp.async instead -> returns 0 (wait with cp.async.wait_group).
__device__ __forceinline__ int warp_stage(unsigned char* buf, unsigned buf_s, unsigned bar_s, unsigned long long src_seg,
                                          unsigned long long rowstride, unsigned long long img_end, int s_lo, int count,
                                          int pitch, int lane, int lr, int lv, int rpp) {
    const unsigned long long first = src_seg + (unsigned long long)s_lo * rowstride;
    const unsigned long long last_end = ((first + (unsigned long long)(count - 1) * rowstride) & ~15ull) + (unsigned long long)pitch;
    if (last_end <= img_end) {
        if (lane == 0) mbar_expect_tx(bar_s, (unsigned)(count * pitch));
        __syncwarp();
        unsigned long long ga = first + (unsigned long long)lane * rowstride;
        unsigned dst = buf_s + lane * pitch;
        for (int r = lane; r < count; r += 32) {
            bulk_g2s(dst, ga & ~15ull, (unsigned)pitch, bar_s);
            ga += 32ull * rowstride;
            dst += 32 * pitch;
        }
        return 1;
    }
    if (lr < rpp) {
        for (int r = lr; r < count; r += rpp) {
            const unsigned long long ga = first + (unsigned long long)r * rowstride;
            const unsigned long long a = (ga & ~15ull) + (unsigned long long)lv * 16ull;
            unsigned char* dst = buf + r * pitch + lv * 16;
            if (a + 16ull <= img_end) {
                cp_async16(dst, (const void*)(uintptr_t)a);
            } else {                                               // last bytes of the image pool
                unsigned int tmp[4] = {0u, 0u, 0u, 0u};
                for (int b = 0; b < 16; ++b)
                    if (a + b < img_end) tmp[b >> 2] |= (unsigned int)(*(const uint8_t*)(uintptr_t)(a + b)) << (8 * (b & 3));
                *reinterpret_cast<uint4*>(dst) = make_uint4(tmp[0], tmp[1], tmp[2], tmp[3]);
            }
        }
    }
    cp_async_commit();
    return 0;
}

// TT = compile-time target size (0: run-time T)
// SWAP = write the planes in R, G, B order from B, G, R sources (cv2.COLOR_BGR2RGB, process_pose.py:206)
template <bool OUT_U8, int TT, bool SWAP>
__global__ void __launch_bounds__(256, 3)
bpc_crop_warp_kernel(const uint8_t* __restrict__ images, int B, int H, int W, const RoiGeom* __restrict__ geom,
                     const float4* __restrict__ xdesc, const float4* __restrict__ ydesc, int32_t* __restrict__ wcount,
                     int R, int Trt, int nslot, uchar4 fill, int swap_rb, const float* __restrict__ lut_g,
                     float* __restrict__ outf, uint8_t* __restrict__ outb) {
    extern __shared__ __align__(128) unsigned char smem[];
    float* lut = reinterpret_cast<float*>(smem);                                 // [3][LUT_STRIDE]: 256 values + the fill value
    const int T = TT ? TT : Trt;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    unsigned char* wbase = smem + LUT_SMEM + wid * WARP_SMEM;         // [2][WARP_BUF] staging, then [2][32] float4 row descriptors
    const unsigned wbase_s = (unsigned)__cvta_generic_to_shared(wbase), lut_s = (unsigned)__cvta_generic_to_shared(smem);

    // see lut_addr(); passed through shared memory so that it stays ONE register (ptxas otherwise re-derives it as window
    // base + constant with an extra add per use)
    if (tid == 0) *reinterpret_cast<volatile unsigned*>(smem + 3 * LUT_STRIDE * 4) = lut_s - 4u * 0x4B000000u;
    const unsigned bar_s = wbase_s + 2 * WARP_BUF + 2 * WARP_DESC;     // eight mbarriers: one per staging buffer / ring slot
    if (lane < 8) mbar_init(bar_s + 8 * lane, 1);
    unsigned ph = 0;                                                      // bit j: parity of the next completion of barrier j
    if (!OUT_U8)
        for (int e = tid; e < 768; e += (int)blockDim.x) lut[(e >> 8) * LUT_STRIDE + (e & 255)] = lut_g[e];
    __syncthreads();
    Out<OUT_U8> out;
    out_init(out, outf, outb, lut, T, swap_rb, fill);
    if (!OUT_U8 && tid < 3) lut[tid * LUT_STRIDE + 256] = out.padf[tid];  // entry 256 = fill: what a lane beside the image looks up
    __syncthreads();
    const unsigned lut_m = *reinterpret_cast<volatile unsigned*>(smem + 3 * LUT_STRIDE * 4);
    const int ds = desc_stride(T), ystride = ydesc_stride(T);
    constexpr bool swap = SWAP;
    const size_t plane = (size_t)T * T;
    const unsigned long long rowstride = (unsigned long long)W * 3ull;
    const unsigned long long img_end = (unsigned long long)(uintptr_t)images + (unsigned long long)B * H * rowstride;
    const float nz = __int_as_float((int)(0x80000000u | (unsigned)fill.w));     // -0.0f: fill.w is 0 at run time
    const u64 nz2 = pack2(nz, nz);
    const long long nitems = (long long)R * nslot;

    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(wcount, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= nitems) break;
        // ROI-major order: a ROI's strips and its (store-only) padding item run at about the same time, which keeps
        // whole output rows together in DRAM and blends store-bound with issue-bound work (padding items last: -8 %)
        const int roi = item / nslot, slot = item - roi * nslot;
        const RoiGeom* gp = geom + roi;
        const int cls = gp->cls;
        if (cls == -1 || cls == 2) continue;
        const int new_w = gp->new_w, new_h = gp->new_h, dx0 = gp->dx, dy0 = gp->dy;

        if (slot == nslot - 1) {
            // ---------------- padding item: rows above / below and column strips left / right ----------------
            if (cls == 0) { out.pad_rows(roi, 0, T, lane, 32); continue; }
            out.pad_rows(roi, 0, dy0, lane, 32);
            out.pad_rows(roi, dy0 + new_h, T, lane, 32);
            // 32-column strips that do not touch the resized image (the others pad their own lanes)
            for (int c = 0; c * 32 < T; ++c) {
                if (c * 32 < dx0 + new_w && c * 32 + 32 > dx0) continue;
                const int x = c * 32 + lane;
                if (x < T)
                    for (int r = 0; r < new_h; ++r) out.pad(roi, dy0 + r, x);
            }
            continue;
        }
        if (cls == 0 || slot * 32 >= dx0 + new_w || slot * 32 + 32 <= dx0) continue;

        // ---------------- output columns [32 slot, 32 slot + 32): full 128-byte lines per plane and row ----------------
        const int x = slot * 32 + lane;
        const int xr = x - dx0;
        const bool active = xr >= 0 && xr < new_w;
        const bool padlane = !active && x < T;
        const float4 xd = xdesc[(size_t)roi * ds + min(max(xr, 0), new_w - 1)];
        const int xs = __float_as_int(xd.w) & 0xffffff;
        const int xn = (cls == 4) ? (__float_as_int(xd.w) >> 24) : 3;     // source pixels read from xs on
        const int xs_min = -warp_max_i32(-xs);
        const int xe_max = warp_max_i32(xs + xn);
        const int seg_bytes = 3 * (xe_max - xs_min);
        const int pitch = ((15 + seg_bytes + 8 + 15) >> 4) << 4;
        const int nv = pitch >> 4;
        const int rpp = 32 / nv, lr = lane / nv, lv = lane - lr * nv;
        const unsigned long long src_seg = gp->src + 3ull * (unsigned long long)xs_min;
        const int mis0 = (int)(src_seg & 15ull), misstep = (int)(rowstride & 15ull);
        const int colc = 3 * (xs - xs_min);
        // byte offset of the lane's first tap in source row s of a buffer staged from row s_lo on: warp_stage() copies every
        // row from the 16-byte boundary below its first byte, so the row's own misalignment moves the tap
        auto tap_off = [&](int s, int s_lo) { return (s - s_lo) * pitch + colc + ((mis0 + s * misstep) & 15); };
        const int rows_fit = WARP_BUF / pitch;
        const double scale_y = gp->scale_y;
        // bh output rows tap at most bh*scale + 2 source rows
        const int bh = max(1, min(32, (int)((double)(rows_fit - 3) / (scale_y < 1.0 ? 1.0 : scale_y))));
        const int nb = (new_h + bh - 1) / bh;
        const float4* ydr = ydesc + (size_t)roi * ystride;
        float* optr = outf + ((size_t)roi * 3 * T + dy0) * T + x;     // (plane 0, current row, column x)
        const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);

        // descriptors of batch b (rows b*bh ..) -> ring k, source rows -> buffer k; returns the first source row
        int bulk_cur = 0, bulk_next = 0;
        auto stage = [&](int b, int k, const float4& yd) -> int {
            const int cnt = min(bh, new_h - b * bh);
            if (lane < cnt) reinterpret_cast<float4*>(wbase + 2 * WARP_BUF + k * WARP_DESC)[lane] = yd;
            int lo, hi;
            if (cls != 3) {
                const int ysn = __float_as_int(yd.w);
                lo = ysn & 0xffffff; hi = lo + (ysn >> 24) - 1;
            } else {
                lo = __float_as_int(yd.w); hi = __float_as_int(yd.z);
            }
            const int s_lo = __shfl_sync(0xffffffffu, lo, 0);
            const int s_hi = __shfl_sync(0xffffffffu, hi, cnt - 1);
            bulk_next = warp_stage(wbase + k * WARP_BUF, wbase_s + k * WARP_BUF, bar_s + 8 * k, src_seg, rowstride, img_end, s_lo,
                                   s_hi - s_lo + 1, pitch, lane, lr, lv, rpp);
            return s_lo;
        };
        auto load_desc = [&](int b) -> float4 {
            const int y = b * bh + lane;
            return (b < nb && y < new_h && lane < bh) ? ydr[y] : zero4;
        };

        if (cls == 4) {
            // ---------------- regime 1, up to 6 taps per axis (2 <= scale <= 5) ----------------
            // Source rows stream through a ring of four slots of G rows (one mbarrier each, three slots in flight while
            // one is read); every row is staged once and its horizontal pass lives in registers, so output rows simply
            // consume rows in order -- no per-output-row batches, which at scale 4 held a single row each.
            const int nt = warp_max_i32(xn);                      // uniform: taps evaluated per source row
            float w[6], c[6];
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                w[k] = (k == 0) ? xd.x : ((k < xn - 1) ? xd.y : ((k == xn - 1) ? xd.z : 0.f));
                c[k] = __fmul_rn(w[k], -8388608.0f);
                asm volatile("" : "+f"(c[k]));
            }
            const int s_first = __float_as_int(ydr[0].w) & 0xffffff;
            const int ysn_last = __float_as_int(ydr[new_h - 1].w);
            const int s_end = (ysn_last & 0xffffff) + (ysn_last >> 24);          // one past the last source row
            const int G = min(32, (2 * WARP_BUF / pitch) >> 2);                  // rows per slot (lane r issues row r)
            const int ngroups = (s_end - s_first + G - 1) / G;
            const unsigned slot_bytes = (unsigned)(G * pitch);
            unsigned bulkmask = 0;
            auto issue = [&](int g) {
                const int j = g & 3, lo = s_first + g * G;
                const int bulk = warp_stage(wbase + j * slot_bytes, wbase_s + j * slot_bytes, bar_s + 8 * j, src_seg, rowstride, img_end,
                                            lo, min(G, s_end - lo), pitch, lane, lr, lv, rpp);
                bulkmask = (bulkmask & ~(1u << j)) | ((unsigned)bulk << j);
            };
            auto wait = [&](int g) {
                const int j = g & 3;
                if ((bulkmask >> j) & 1u) { mbar_wait(bar_s + 8 * j, (ph >> j) & 1u); ph ^= 1u << j; }
                else cp_async_wait_all();
                __syncwarp();
            };
            __syncwarp();                                   // previous item finished with the buffers
            for (int g = 0; g < min(4, ngroups); ++g) issue(g);
            wait(0);
            int gi = 0, gend = s_first + G;                 // current group and one past its last row
            int crow = -1;
            u64 hc01 = 0ull;
            float hc2 = 0.f;
            auto strip = [&](auto nt_c) {
                constexpr int NT = decltype(nt_c)::value;
                auto hrow = [&](int row) {
                    while (row >= gend) {
                        __syncwarp();                       // every lane is done with slot gi & 3
                        if (gi + 4 < ngroups) issue(gi + 4);
                        ++gi;
                        wait(gi);
                        gend += G;
                    }
                    const int a = tap_off(row, gend - G);
                    h_area_n<NT>(wbase_s + (unsigned)(gi & 3) * slot_bytes + (a & ~3), (a & 3) * 8, w, c, hc01, hc2);
                };
                float4 d = ydr[0];
                for (int y = 0; y < new_h; ++y) {
                    const float4 dn = ydr[min(y + 1, new_h - 1)];
                    const int ysn = __float_as_int(d.w);
                    const int ys = ysn & 0xffffff, n = ysn >> 24;
                    if (ys != crow) hrow(ys);                // else: the previous output row ended on this source row
                    u64 acc01 = fprod2(pack2(d.x, d.x), hc01, nz2);
                    float acc2 = __fmul_rn(d.x, hc2);
                    for (int t = 1; t < n; ++t) {
                        hrow(ys + t);
                        const float beta = (t == n - 1) ? d.z : d.y;
                        acc01 = fadd2(acc01, fprod2(pack2(beta, beta), hc01, nz2));
                        acc2 = __fadd_rn(acc2, __fmul_rn(beta, hc2));
                    }
                    crow = ys + n - 1;
                    if (active) {
                        float a0f, a1f;
                        unpack2(acc01, a0f, a1f);
                        if (OUT_U8) {
                            out.px(roi, dy0 + y, x, round_u8(a0f), round_u8(a1f), round_u8(acc2));
                        } else {
                            const unsigned l0 = lut_addr(a0f, lut_m), l1 = lut_addr(a1f, lut_m), l2 = lut_addr(acc2, lut_m);
                            optr[0] = lds_f32(swap ? l2 : l0);
                            optr[plane] = lds_f32(l1 + 4 * LUT_STRIDE);
                            optr[2 * plane] = lds_f32((swap ? l0 : l2) + 8 * LUT_STRIDE);
                            optr += T;
                        }
                    } else if (padlane) {
                        out.pad(roi, dy0 + y, x);
                    }
                    d = dn;
                }
            };
            if (nt <= 4) strip(std::integral_constant<int, 4>{});
            else if (nt == 5) strip(std::integral_constant<int, 5>{});
            else strip(std::integral_constant<int, 6>{});
            continue;
        }

        __syncwarp();                                   // previous item finished with the buffers
        int s_lo_cur = stage(0, 0, load_desc(0));
        bulk_cur = bulk_next;
        float4 ydn = load_desc(1);
        int s_lo_next = 0;

        if (cls == 1) {
            ColW cw;
            cw.set(xd.x, xd.y, xd.z);
            int crow = -1;
            u64 hc01 = 0ull;
            float hc2 = 0.f;
            unsigned roff = 0;                                // element offset of the current output row from optr
            for (int b = 0; b < nb; ++b) {
                const int k = b & 1;
                if (bulk_cur) {
                    mbar_wait(bar_s + 8 * k, (ph >> k) & 1u); ph ^= 1u << k;
                } else {
                    cp_async_wait_all();
                }
                __syncwarp();
                if (b + 1 < nb) s_lo_next = stage(b + 1, k ^ 1, ydn);
                ydn = load_desc(b + 2);
                const unsigned cur = wbase_s + k * WARP_BUF, ring = wbase_s + 2 * WARP_BUF + k * WARP_DESC;
                const int y0 = b * bh, cnt = min(bh, new_h - y0);
                if (active) {
                    float4 dnx = lds_f4(ring);
                    for (int r = 0; r < cnt; ++r) {
                        const float4 d = dnx;
                        dnx = lds_f4(ring + (r + 1) * 16);          // next row's descriptor in flight behind this row's arithmetic
                        const int ysn = __float_as_int(d.w);
                        const int ys = ysn & 0xffffff, n = ysn >> 24;
                        const int a = tap_off(ys, s_lo_cur);
                        if (ys != crow) h_area3(cur + (a & ~3), (a & 3) * 8, cw, hc01, hc2);
                        u64 acc01 = fprod2(pack2(d.x, d.x), hc01, nz2);
                        float acc2 = __fmul_rn(d.x, hc2);
                        if (n > 1) {
                            const int a1 = tap_off(ys + 1, s_lo_cur);
                            h_area3(cur + (a1 & ~3), (a1 & 3) * 8, cw, hc01, hc2);
                            acc01 = fadd2(acc01, fprod2(pack2(d.y, d.y), hc01, nz2));
                            acc2 = __fadd_rn(acc2, __fmul_rn(d.y, hc2));
                        }
                        if (n > 2) {
                            const int a2 = tap_off(ys + 2, s_lo_cur);
                            h_area3(cur + (a2 & ~3), (a2 & 3) * 8, cw, hc01, hc2);
                            acc01 = fadd2(acc01, fprod2(pack2(d.z, d.z), hc01, nz2));
                            acc2 = __fadd_rn(acc2, __fmul_rn(d.z, hc2));
                        }
                        crow = ys + n - 1;
                        float a0f, a1f;
                        unpack2(acc01, a0f, a1f);
                        if (OUT_U8) {
                            out.px(roi, dy0 + y0 + r, x, round_u8(a0f), round_u8(a1f), round_u8(acc2));
                        } else {
                            // bits(v + 2^23) = 0x4B000000 + cvRound(v): the LUT address is one multiply-add away
                            const unsigned l0 = lut_addr(a0f, lut_m), l1 = lut_addr(a1f, lut_m), l2 = lut_addr(acc2, lut_m);
                            float* o = optr + roff;               // fresh address registers per row: no wait on the previous row's stores
                            o[0] = lds_f32(swap ? l2 : l0);
                            o[plane] = lds_f32(l1 + 4 * LUT_STRIDE);
                            o[2 * plane] = lds_f32((swap ? l0 : l2) + 8 * LUT_STRIDE);
                            roff += (unsigned)T;
                        }
                    }
                } else if (padlane) {
                    for (int r = 0; r < cnt; ++r) out.pad(roi, dy0 + y0 + r, x);
                }
                s_lo_cur = s_lo_next;
                bulk_cur = bulk_next;
            }
        } else {
            const int xw0 = __float_as_int(xd.x), xw1 = __float_as_int(xd.y);
            int rowA = -1, rowB = -1;
            int HA[3] = {0, 0, 0}, HB[3] = {0, 0, 0};
            for (int b = 0; b < nb; ++b) {
                const int k = b & 1;
                if (bulk_cur) {
                    mbar_wait(bar_s + 8 * k, (ph >> k) & 1u); ph ^= 1u << k;
                } else {
                    cp_async_wait_all();
                }
                __syncwarp();
                if (b + 1 < nb) s_lo_next = stage(b + 1, k ^ 1, ydn);
                ydn = load_desc(b + 2);
                const unsigned cur = wbase_s + k * WARP_BUF, ring = wbase_s + 2 * WARP_BUF + k * WARP_DESC;
                const int y0 = b * bh, cnt = min(bh, new_h - y0);
                if (active) {
                    for (int r = 0; r < cnt; ++r) {
                        const float4 d = lds_f4(ring + r * 16);
                        const int b0 = __float_as_int(d.x), b1 = __float_as_int(d.y);
                        const int sy0 = __float_as_int(d.w), sy1 = __float_as_int(d.z);
                        if (sy0 != rowA) {
                            if (sy0 == rowB) { HA[0] = HB[0]; HA[1] = HB[1]; HA[2] = HB[2]; }
                            else {
                                const int a = tap_off(sy0, s_lo_cur);
                                h_lin(cur + (a & ~3), (a & 3) * 8, xw0, xw1, HA);
                            }
                            rowA = sy0;
                        }
                        if (sy1 != rowB) {
                            if (sy1 == rowA) { HB[0] = HA[0]; HB[1] = HA[1]; HB[2] = HA[2]; }
                            else {
                                const int a = tap_off(sy1, s_lo_cur);
                                h_lin(cur + (a & ~3), (a & 3) * 8, xw0, xw1, HB);
                            }
                            rowB = sy1;
                        }
                        int o[3];
#pragma unroll
                        for (int c = 0; c < 3; ++c) o[c] = ((((b0 * HA[c]) >> 16) + ((b1 * HB[c]) >> 16) + 2) >> 2) & 255;
                        if (OUT_U8) {
                            out.px(roi, dy0 + y0 + r, x, o[0], o[1], o[2]);
                        } else {
                            optr[0] = lds_f32(lut_s + 4 * (swap ? o[2] : o[0]));
                            optr[plane] = lds_f32(lut_s + 4 * LUT_STRIDE + 4 * o[1]);
                            optr[2 * plane] = lds_f32(lut_s + 8 * LUT_STRIDE + 4 * (swap ? o[0] : o[2]));
                            optr += T;
                        }
                    }
                } else if (padlane) {
                    for (int r = 0; r < cnt; ++r) out.pad(roi, dy0 + y0 + r, x);
                }
                s_lo_cur = s_lo_next;
                bulk_cur = bulk_next;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// generic kernel: any regime / scale, persistent CTAs over (ROI, band) items of the generic list
// ------------------------------------------------------------------------------------------------------
template <bool OUT_U8, bool BF16>
__device__ void crop_generic_band(unsigned char* raw, YDesc* yd, const Out<OUT_U8, BF16>& out, const RoiGeom& g, int roi, int band,
                                  const uint8_t* __restrict__ images, int B, int H, int W, int T, int tid, int nth) {
    const int x = tid;
    const bool incol = x < T;
    const int row0 = band * CROP_BAND, row1 = min(T, row0 + CROP_BAND);
    const int regime = g.regime;
    const int dy0 = g.dy, new_h = g.new_h, new_w = g.new_w, dx0 = g.dx;
    const int ya = max(row0, dy0) - dy0, yb = min(row1, dy0 + new_h) - dy0;
    out.pad_rows(roi, row0, min(row1, dy0), tid, nth);
    out.pad_rows(roi, max(row0, dy0 + new_h), row1, tid, nth);
    if (ya >= yb) return;                                            // uniform

    const int w = g.w, h = g.h;
    if (tid < yb - ya) {
        YDesc d;
        const int yr = ya + tid;
        if (regime == 1) {
            area_taps(yr, g.scale_y, h, d.start, d.n, d.bf, d.bm, d.bl, d.flags);
        } else if (regime == 2) {
            d.start = yr * g.isy; d.n = g.isy; d.bf = d.bm = d.bl = 1.f; d.flags = 0;
        } else {
            int s0, b0, b1, edge;
            linear_coef(yr, g.scale_y, g.inv_y, h, s0, b0, b1, edge);
            d.start = s0; d.n = min(s0 + 1, h - 1);
            d.bf = __int_as_float(b0); d.bm = __int_as_float(b1); d.bl = 0.f; d.flags = 0;
        }
        yd[tid] = d;
    }
    const int xr = x - dx0;
    const bool active = incol && xr >= 0 && xr < new_w;
    int xs = 0, xn = 0, xflags = 0, xw0 = 0, xw1 = 0, xedge = 0;
    float af = 0.f, am = 0.f, al = 0.f;
    if (active) {
        if (regime == 1) area_taps(xr, g.scale_x, w, xs, xn, af, am, al, xflags);
        else if (regime == 2) { xs = xr * g.isx; xn = g.isx; }
        else linear_coef(xr, g.scale_x, g.inv_x, w, xs, xw0, xw1, xedge);
    }
    __syncthreads();

    const int s_lo = yd[0].start;
    const int s_hi = (regime == 3) ? yd[yb - ya - 1].n : (yd[yb - ya - 1].start + yd[yb - ya - 1].n - 1);
    const int pitch = ((3 * w + 15 + 15) / 16) * 16;
    const int rows_fit = CROP_RAW_BYTES / pitch;
    const unsigned long long src0 = g.src;
    const unsigned long long rowstride = (unsigned long long)W * 3ull;
    const unsigned long long img_end = (unsigned long long)(uintptr_t)images + (unsigned long long)B * H * rowstride;
    const int nvec = pitch >> 4;
    const int lane = tid & 31, wid = tid >> 5, nwarps = nth >> 5;

    int yr = ya, t = 0;                      // streaming state, uniform across the CTA except for x
    float acc[3] = {0.f, 0.f, 0.f};
    int iacc[3] = {0, 0, 0};
    int cacheA = -1, cacheB = -1;
    float hA[3] = {0.f, 0.f, 0.f};
    int HA[3] = {0, 0, 0}, HB[3] = {0, 0, 0};

    int chunk = s_lo;
    while (yr < yb) {
        const int rows = min(rows_fit, s_hi - chunk + 1);
        __syncthreads();
        for (int r = wid; r < rows; r += nwarps) {
            const unsigned long long ga = src0 + (unsigned long long)(chunk + r) * rowstride;
            const unsigned long long al16 = ga & ~15ull;
            const int need = (int)(ga - al16) + 3 * w;
            for (int v = lane; v < nvec; v += 32) {
                if (v * 16 >= need) break;
                const unsigned long long a = al16 + (unsigned long long)v * 16ull;
                uint4 q;
                if (a + 16ull <= img_end) {
                    q = ld_nc_v4((const void*)(uintptr_t)a);
                } else {
                    unsigned int tmp[4] = {0u, 0u, 0u, 0u};
                    for (int b = 0; b < 16; ++b)
                        if (a + b < img_end) tmp[b >> 2] |= (unsigned int)(*(const uint8_t*)(uintptr_t)(a + b)) << (8 * (b & 3));
                    q = make_uint4(tmp[0], tmp[1], tmp[2], tmp[3]);
                }
                *reinterpret_cast<uint4*>(raw + (size_t)r * pitch + (size_t)v * 16) = q;
            }
        }
        __syncthreads();
        const int chunk_end = chunk + rows;
        auto rowptr = [&](int sy) -> const uint8_t* {
            const unsigned long long ga = src0 + (unsigned long long)sy * rowstride;
            return raw + (size_t)(sy - chunk) * pitch + (int)(ga & 15ull);
        };

        if (regime == 3) {
            while (yr < yb) {
                const YDesc d = yd[yr - ya];
                const int sy0 = d.start, sy1 = d.n;
                if (sy1 >= chunk_end) break;
                if (active) {
                    if (cacheA != sy0) {
                        if (cacheB == sy0) { HA[0] = HB[0]; HA[1] = HB[1]; HA[2] = HB[2]; }
                        else {
                            const uint8_t* p = rowptr(sy0) + 3 * xs;
                            for (int c = 0; c < 3; ++c) HA[c] = xedge ? (int)p[c] * 2048 : (int)p[c] * xw0 + (int)p[3 + c] * xw1;
                        }
                        cacheA = sy0;
                    }
                    if (cacheB != sy1) {
                        if (sy1 == sy0) { HB[0] = HA[0]; HB[1] = HA[1]; HB[2] = HA[2]; }
                        else {
                            const uint8_t* p = rowptr(sy1) + 3 * xs;
                            for (int c = 0; c < 3; ++c) HB[c] = xedge ? (int)p[c] * 2048 : (int)p[c] * xw0 + (int)p[3 + c] * xw1;
                        }
                        cacheB = sy1;
                    }
                    const int b0 = __float_as_int(d.bf), b1 = __float_as_int(d.bm);
                    int o[3];
                    for (int c = 0; c < 3; ++c)
                        o[c] = ((((b0 * (HA[c] >> 4)) >> 16) + ((b1 * (HB[c] >> 4)) >> 16) + 2) >> 2) & 255;
                    out.px(roi, dy0 + yr, x, o[0], o[1], o[2]);
                } else if (incol) {
                    out.pad(roi, dy0 + yr, x);
                }
                ++yr;
            }
            if (yr < yb) chunk = yd[yr - ya].start;
        } else {
            while (yr < yb) {
                const YDesc d = yd[yr - ya];
                const int sy = d.start + t;
                if (sy >= chunk_end) break;
                if (active) {
                    const uint8_t* p = rowptr(sy) + 3 * xs;
                    if (regime == 1) {
                        if (cacheA != sy) {
                            float s0 = 0.f, s1 = 0.f, s2 = 0.f;
                            for (int k = 0; k < xn; ++k) {
                                const float a = (k == 0 && (xflags & 1)) ? af : ((k == xn - 1 && (xflags & 2)) ? al : am);
                                s0 = __fadd_rn(s0, __fmul_rn((float)p[3 * k + 0], a));
                                s1 = __fadd_rn(s1, __fmul_rn((float)p[3 * k + 1], a));
                                s2 = __fadd_rn(s2, __fmul_rn((float)p[3 * k + 2], a));
                            }
                            hA[0] = s0; hA[1] = s1; hA[2] = s2;
                            cacheA = sy;
                        }
                        const float beta = (t == 0 && (d.flags & 1)) ? d.bf : ((t == d.n - 1 && (d.flags & 2)) ? d.bl : d.bm);
                        for (int c = 0; c < 3; ++c) {
                            const float term = __fmul_rn(beta, hA[c]);
                            acc[c] = (t == 0) ? term : __fadd_rn(acc[c], term);
                        }
                    } else {
                        if (t == 0) { iacc[0] = 0; iacc[1] = 0; iacc[2] = 0; }
                        for (int k = 0; k < xn; ++k) {
                            iacc[0] += p[3 * k + 0]; iacc[1] += p[3 * k + 1]; iacc[2] += p[3 * k + 2];
                        }
                    }
                }
                ++t;
                if (t == d.n) {
                    if (active) {
                        int o[3];
                        if (regime == 1) {
                            for (int c = 0; c < 3; ++c) o[c] = min(255, max(0, __float2int_rn(acc[c])));
                        } else if (g.isx == 2 && g.isy == 2) {
                            for (int c = 0; c < 3; ++c) o[c] = (iacc[c] + 2) >> 2;
                        } else {
                            const float sc = __fdiv_rn(1.f, (float)(g.isx * g.isy));
                            for (int c = 0; c < 3; ++c) o[c] = min(255, max(0, __float2int_rn(__fmul_rn(__int2float_rn(iacc[c]), sc))));
                        }
                        out.px(roi, dy0 + yr, x, o[0], o[1], o[2]);
                    } else if (incol) {
                        out.pad(roi, dy0 + yr, x);
                    }
                    ++yr; t = 0;
                }
            }
            if (yr < yb) chunk = yd[yr - ya].start + t;
        }
    }
}

template <bool OUT_U8, int NTH, bool BF16 = false>
__global__ void __launch_bounds__(NTH)
bpc_crop_generic_kernel(const uint8_t* __restrict__ images, int B, int H, int W, const RoiGeom* __restrict__ geom,
                        const int32_t* __restrict__ glist, const int32_t* __restrict__ gcount, int T, int nbands,
                        uchar4 fill, int swap_rb, const float* __restrict__ lut_g, float* __restrict__ outf, uint8_t* __restrict__ outb) {
    extern __shared__ __align__(16) unsigned char raw[];
    __shared__ RoiGeom g;
    __shared__ YDesc yd[CROP_BAND];
    __shared__ float lut[OUT_U8 ? 1 : 3 * LUT_STRIDE];
    const int tid = threadIdx.x, nth = blockDim.x;
    const long long items = (long long)(*gcount) * nbands;
    if (blockIdx.x >= items) return;
    if (!OUT_U8)
        for (int e = tid; e < 768; e += nth) lut[(e >> 8) * LUT_STRIDE + (e & 255)] = lut_g[e];
    __syncthreads();
    Out<OUT_U8, BF16> out;
    out_init(out, outf, outb, lut, T, swap_rb, fill);
    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        const int roi = glist[item / nbands], band = (int)(item % nbands);
        __syncthreads();
        if (tid == 0) g = geom[roi];
        __syncthreads();
        crop_generic_band<OUT_U8, BF16>(raw, yd, out, g, roi, band, images, B, H, W, T, tid, nth);
    }
}

__global__ void bpc_lut_kernel(float m0, float m1, float m2, float s0, float s1, float s2, float* __restrict__ lut) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 768) return;
    const int c = t >> 8, v = t & 255;
    const float mean = c == 0 ? m0 : (c == 1 ? m1 : m2);
    const float sd = c == 0 ? s0 : (c == 1 ? s1 : s2);
    // to_tensor: float(v) / 255 ; normalize: (x - mean) / std -- float32, true divisions
    lut[t] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)v, 255.f), mean), sd);
}

// workspace: geom[R] | xdesc[R][ds] | ydesc[R][ydesc_stride(T)] | counters[16] | glist[R] | list1[R]    (ds = desc_stride(T), float4 records)
static size_t ws_off_xdesc(int R) { return (((size_t)R * sizeof(RoiGeom)) + 15) & ~(size_t)15; }
static size_t ws_off_ydesc(int R, int T) { return ws_off_xdesc(R) + (size_t)R * desc_stride(T) * sizeof(float4); }
static size_t ws_off_count(int R, int T) { return ws_off_ydesc(R, T) + (size_t)R * ydesc_stride(T) * sizeof(float4); }
static size_t crop_workspace_bytes(int R, int T) { return ws_off_count(R, T) + 64 + 2 * (size_t)R * sizeof(int32_t) + 64; }

template <bool OUT_U8, bool BF16 = false>
static int launch_crop(const uint8_t* images, int B, int H, int W, const int32_t* rois, int R, const int32_t* n_rois_dev,
                       int roi_first, int T, const uint8_t* fill, int swap_rb, const float* lut, float* outf, uint8_t* outb,
                       int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
    if (R < 0 || B < 1 || H < 1 || W < 1 || T < 1 || T > BPC_MAX_TARGET || !fill) return BPC_EINVAL;
    if (R > 0 && (!images || !rois || !workspace || (!OUT_U8 && (!lut || !outf)) || (OUT_U8 && !outb))) return BPC_EINVAL;
    if (((uintptr_t)images & 15) != 0 || ((uintptr_t)workspace & 15) != 0) return BPC_EALIGN;
    if (R == 0) return BPC_OK;
    if (workspace_bytes < crop_workspace_bytes(R, T)) return BPC_EWORKSPACE;
    const int nslot = (T + 31) / 32 + 1;
    if ((long long)R * nslot > 0x7fffffffLL) return BPC_ETOOBIG;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* wsb = (unsigned char*)workspace;
    RoiGeom* geom = (RoiGeom*)wsb;
    float4* xdesc = (float4*)(wsb + ws_off_xdesc(R));
    float4* ydesc = (float4*)(wsb + ws_off_ydesc(R, T));
    int32_t* gcount = (int32_t*)(wsb + ws_off_count(R, T));   // [0] generic-list length, [4] warp-item counter, [8] CTA-list length, [9] 1 if that list was reordered, [12] its work counter
    int32_t* wcount = gcount + 4;
    int32_t* glist = gcount + 16;
    int32_t* list1 = glist + R;
    cudaError_t e = cudaMemsetAsync(gcount, 0, 64, st);
    if (e != cudaSuccess) return (int)e;
    // the CTA kernel stages full-width 2-D TMA boxes: a 16-byte row pitch, at most eight strips, its widest box inside the pool rows
    const long long pitch = (long long)W * 3;
    const bool use_cta = pitch % 16 == 0 && pitch >= WARP_MAX_PITCH && T <= CTA_MAX_T && pitch >= cta_pitch_max(T);
    if (BF16 && !use_cta) return BPC_EUNSUPPORTED;       // the bfloat16 output exists on the CTA kernel's path only
    bpc_crop_prep_kernel<<<R, PREP_THREADS, 0, st>>>(images, B, H, W, rois, n_rois_dev, roi_first, T, use_cta ? 1 : 0, geom, xdesc, ydesc,
                                            glist, gcount, status, list1);
    BPC_LAUNCH_CHECK();
    const uchar4 f4 = make_uchar4(fill[0], fill[1], fill[2], 0);
    if (use_cta) {                                        // every fast-class crop is on the CTA kernel's list
        bpc_crop_order_kernel<<<ORDER_CTAS, ORDER_THREADS, 0, st>>>(images, B, H, W, geom, list1, gcount, glist);
        BPC_LAUNCH_CHECK();
        const int rc = crop_cta_launch(OUT_U8 ? 1 : (BF16 ? 2 : 0), images, B, H, W, geom, xdesc, ydesc, list1, gcount, R, T, f4, swap_rb, lut,
                                       outf, outb, st);
        if (rc != BPC_OK) return rc;
    } else {
        // the uint8 entry point never swaps channels and keeps T a run-time value: one variant
        auto fn = bpc_crop_warp_kernel<OUT_U8, 0, false>;
        if constexpr (!OUT_U8) {
            const bool sw = swap_rb != 0;
            if (T == 224) fn = sw ? bpc_crop_warp_kernel<false, 224, true> : bpc_crop_warp_kernel<false, 224, false>;
            else if (T == 256) fn = sw ? bpc_crop_warp_kernel<false, 256, true> : bpc_crop_warp_kernel<false, 256, false>;
            else if (sw) fn = bpc_crop_warp_kernel<false, 0, true>;
        }
        // the same constant on every call: idempotent, so concurrent callers cannot interleave set(small) / launch(large)
        e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, WARPK_SMEM);
        if (e != cudaSuccess) return (int)e;
        const int cta_threads = 256;
        const long long nitems = (long long)R * nslot;
        const long long want = (nitems + WARPK_WARPS - 1) / WARPK_WARPS;
        int dev = 0, sms = 148, per_sm = 3;                     // persistent grid: every resident CTA slot, no more
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, cta_threads, WARPK_SMEM) != cudaSuccess || per_sm < 1) per_sm = 1;
        const long long slots = (long long)sms * per_sm;
        const int grid = (int)(want < slots ? want : slots);
        fn<<<grid, cta_threads, WARPK_SMEM, st>>>(images, B, H, W, geom, xdesc, ydesc, wcount, R, T, nslot, f4, swap_rb, lut, outf, outb);
        BPC_LAUNCH_CHECK();
    }
    const int nbands = (T + CROP_BAND - 1) / CROP_BAND;
    const long long max_items = (long long)R * nbands;
    const int grid = (int)(max_items < 148 * 2 ? max_items : 148 * 2);
    const int threads = ((T + 31) / 32) * 32;                   // one thread per output column
    auto gfn = bpc_crop_generic_kernel<OUT_U8, 256, BF16>;
    if constexpr (!BF16)                                        // bfloat16 runs beside the CTA kernel only: T <= 256
        if (threads > 256) gfn = bpc_crop_generic_kernel<OUT_U8, 1024>;
    e = cudaFuncSetAttribute(gfn, cudaFuncAttributeMaxDynamicSharedMemorySize, CROP_RAW_BYTES);
    if (e != cudaSuccess) return (int)e;
    gfn<<<grid, threads, CROP_RAW_BYTES, st>>>(images, B, H, W, geom, glist, gcount, T, nbands, f4, swap_rb, lut, outf, outb);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

}  // namespace bpc

using namespace bpc;

extern "C" size_t bpc_roi_crop_workspace_bytes(int R, int T) { return (R < 0 || T < 1 || T > BPC_MAX_TARGET) ? 0 : crop_workspace_bytes(R, T); }

extern "C" int bpc_roi_crop(const uint8_t* images, int B, int H, int W, const int32_t* rois, int R,
                            const int32_t* n_rois_dev, int roi_first, int T, const uint8_t* fill, int swap_rb,
                            const float* lut, float* out, int32_t* status, void* workspace, size_t workspace_bytes,
                            void* stream) {
    if (((uintptr_t)out & 15) != 0) return BPC_EALIGN;
    return launch_crop<false>(images, B, H, W, rois, R, n_rois_dev, roi_first, T, fill, swap_rb, lut, out, nullptr, status,
                              workspace, workspace_bytes, stream);
}

extern "C" int bpc_roi_crop_bf16(const uint8_t* images, int B, int H, int W, const int32_t* rois, int R,
                                 const int32_t* n_rois_dev, int roi_first, int T, const uint8_t* fill, int swap_rb,
                                 const float* lut, void* out, int32_t* status, void* workspace, size_t workspace_bytes,
                                 void* stream) {
    if (((uintptr_t)out & 15) != 0) return BPC_EALIGN;
    return launch_crop<false, true>(images, B, H, W, rois, R, n_rois_dev, roi_first, T, fill, swap_rb, lut, (float*)out, nullptr, status,
                                    workspace, workspace_bytes, stream);
}

extern "C" int bpc_roi_crop_u8(const uint8_t* images, int B, int H, int W, const int32_t* rois, int R,
                               const int32_t* n_rois_dev, int roi_first, int T, const uint8_t* fill, uint8_t* out,
                               int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
    return launch_crop<true>(images, B, H, W, rois, R, n_rois_dev, roi_first, T, fill, 0, nullptr, nullptr, out, status,
                             workspace, workspace_bytes, stream);
}

extern "C" int bpc_normalise_lut(const float* mean, const float* std_, float* lut, void* stream) {
    if (!mean || !std_ || !lut) return BPC_EINVAL;
    bpc_lut_kernel<<<3, 256, 0, (cudaStream_t)stream>>>(mean[0], mean[1], mean[2], std_[0], std_[1], std_[2], lut);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}
