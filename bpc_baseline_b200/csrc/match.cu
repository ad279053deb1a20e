// Geometry kernels of libbpc_b200: fundamental matrices, cost tensor, assignment, triangulation.
//
// bpc_match_triangulate = PoseEstimator._match (bpc/inference/process_pose.py:144-188) for a batch of
// independent scenes, one CTA per scene, everything in shared memory / registers:
//   phase 0  F12/F13/F23 (camera_utils.py:23-46), P = K @ RT[:3] (process_pose.py:91), two normalised
//            epipolar lines per detection and camera pair (epipolar_matching.py:13-23);
//   phase 1  one warp per third-camera detection k: exact argmin over the N*M (i, j) pairs of the VIRTUAL
//            cost tensor (epipolar_matching.py:83-98 is never materialised), pruned with
//            sum >= e13[i,k] and sum >= e23[j,k];
//   phase 2  SciPy-exact assignment (lsap.cuh): rows whose argmin column is still free are immediate
//            sinks; conflicts and exact ties run the full shortest-augmenting-path search;
//   phase 3  threshold (epipolar_matching.py:110-111), sort by (cost, r) (process_pose.py:183), DLT
//            triangulation and reprojection error per match, one thread each.
#include "geometry.cuh"
#include "lsap.cuh"

namespace bpc {

// ------------------------------------------------------------------------------------------------------
// cost accessors for the assignment
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_min_d(double v);
__device__ __forceinline__ int warp_min_i(int v);

struct VirtualCost {            // cost.reshape(N*M, P) of the epipolar cost tensor
    const Scene* sc;
    int transposed;             // 1: rows = k, cols = r = i*M + j   (N*M > P, SciPy transposes)
    // per-warp scratch for the pruned column scan (the phase-1 buffers, free during the assignment); null = scan everything
    double* wa; double* wb; short* wil; short* wjl;
    __device__ __forceinline__ double cost(int row, int col) const {
        const int r = transposed ? col : row;
        const int k = transposed ? row : col;
        const int i = (int)(((unsigned long long)(unsigned)r * sc->m_magic) >> 40), j = r - i * sc->M;
        return (double)sc->cost(i, j, k);
    }
    __device__ void scan_unassigned(const LsapState& st, int t, int nov, Cand& best, int nthreads, int tid) const;
};

struct ExplicitCost {           // dense float32 [N*M][P]
    const float* c;
    int P;
    int transposed;
    __device__ __forceinline__ double cost(int row, int col) const {
        const int r = transposed ? col : row;
        const int k = transposed ? row : col;
        return (double)c[(size_t)r * P + k];
    }
    __device__ __forceinline__ void scan_unassigned(const LsapState& st, int t, int nov, Cand& best, int nthreads, int tid) const {
        lsap_scan_unassigned_full(st, *this, t, nov, best, nthreads, tid);
    }
};

// ------------------------------------------------------------------------------------------------------
// phase 1: per-row argmin of the virtual cost tensor (transposed case), one warp per row k
// ------------------------------------------------------------------------------------------------------
struct RowMin {
    float* cmin;   // [P] float32 cost of the best column
    int* rlo;      // [P] lowest column index r attaining it
    int* cnt;      // [P] number of columns attaining it (float32 equality); 0 when the minimum is +inf
};

__device__ __forceinline__ double warp_min_d(double v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = fmin(v, shfl_xor_d(v, m));
    return v;
}
__device__ __forceinline__ int warp_min_i(int v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, m));
    return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    return v;
}

// scratch per warp: a[Dmax], b[Dmax] doubles, il[Dmax], jl[Dmax] int16
__device__ void row_argmin(const Scene& sc, int k, double* sa, double* sb, short* il, short* jl, RowMin out) {
    const int lane = lane_id();
    const int N = sc.N, M = sc.M;
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    // a_i = e13[i,k], b_j = e23[j,k]
    double amin = INF, bmin = INF;
    int i0 = 0x7fffffff, j0 = 0x7fffffff;
    for (int i = lane; i < N; i += 32) {
        const double a = sc.e13(i, k);
        sa[i] = a;
        if (a < amin) { amin = a; i0 = i; }
    }
    for (int j = lane; j < M; j += 32) {
        const double b = sc.e23(j, k);
        sb[j] = b;
        if (b < bmin) { bmin = b; j0 = j; }
    }
    const double wa = warp_min_d(amin), wb = warp_min_d(bmin);
    i0 = warp_min_i(amin == wa ? i0 : 0x7fffffff);
    j0 = warp_min_i(bmin == wb ? j0 : 0x7fffffff);
    if (i0 >= N) i0 = 0;       // all-NaN guards
    if (j0 >= M) j0 = 0;
    __syncwarp();
    // seed an upper bound: first the sum at (i0, j0) itself (for a clean scene that already is the minimum and prunes
    // nearly every candidate below), then the row / column through the individually best i and j
    double best = dadd(dadd(sc.e12(i0, j0), sa[i0]), sb[j0]);
    for (int j = lane; j < M; j += 32)
        if (sb[j] <= best) best = fmin(best, dadd(dadd(sc.e12(i0, j), sa[i0]), sb[j]));
    for (int i = lane; i < N; i += 32)
        if (sa[i] <= best) best = fmin(best, dadd(dadd(sc.e12(i, j0), sa[i]), sb[j0]));
    best = warp_min_d(best);
    // every (i, j) whose float32 cost can equal the minimum has sum <= bound, hence a_i, b_j <= bound
    // (sum = fl(fl(e12 + a) + b) >= max(a, b) because rounding is monotone and e12 >= 0)
    const double bound = dadd(dmul(best, 1.0 + 2.384185791015625e-07), 1e-37);
    int nI = 0, nJ = 0;
    for (int base = 0; base < N; base += 32) {
        const int i = base + lane;
        const bool p = i < N && sa[i] <= bound;
        const unsigned m = __ballot_sync(0xffffffffu, p);
        if (p) il[nI + __popc(m & ((1u << lane) - 1))] = (short)i;
        nI += __popc(m);
    }
    for (int base = 0; base < M; base += 32) {
        const int j = base + lane;
        const bool p = j < M && sb[j] <= bound;
        const unsigned m = __ballot_sync(0xffffffffu, p);
        if (p) jl[nJ + __popc(m & ((1u << lane) - 1))] = (short)j;
        nJ += __popc(m);
    }
    __syncwarp();
    const int npair = nI * nJ;
    double smin = INF;
    for (int q = lane; q < npair; q += 32) {
        const int ii = q / nJ, jj = q - ii * nJ;
        const int i = il[ii], j = jl[jj];
        smin = fmin(smin, dadd(dadd(sc.e12(i, j), sa[i]), sb[j]));
    }
    smin = warp_min_d(smin);
    const float cmin = cost_from_sum(smin);
    int cnt = 0, rlo = 0x7fffffff;
    for (int q = lane; q < npair; q += 32) {
        const int ii = q / nJ, jj = q - ii * nJ;
        const int i = il[ii], j = jl[jj];
        const double s = dadd(dadd(sc.e12(i, j), sa[i]), sb[j]);
        if (s <= bound && cost_from_sum(s) == cmin) { ++cnt; rlo = min(rlo, i * M + j); }
    }
    cnt = warp_sum_i(cnt);
    rlo = warp_min_i(rlo);
    // a +inf minimum: every column may round to +inf, not only those below the bound, so the count is unknown (0 = not
    // an immediate sink; the augmenting-path search then finds no finite path, and SciPy reports infeasible)
    if (!(cmin < __int_as_float(0x7f800000))) cnt = 0;
    if (lane == 0) { out.cmin[k] = cmin; out.cnt[k] = cnt; out.rlo[k] = rlo; }
    __syncwarp();
}

// ------------------------------------------------------------------------------------------------------
// phase 2 helper: the Dijkstra step's scan over the (up to 40 000) unassigned columns, pruned
// ------------------------------------------------------------------------------------------------------
// The step needs the unassigned column with the lowest label min_a r_a(col), r_a = (cm[a] + cost(k_a, col)) - cu[a],
// ties resolved by SciPy's scan position.  r_a is monotone in the cost and cost(k, (i, j)) = f32(sum / 3) with
// sum >= e13[i, k] and sum >= e23[j, k] (phase 1), so for each chain row a one warp (i) evaluates a_i = e13[i, k_a] and
// b_j = e23[j, k_a], (ii) takes an upper bound on the minimum from the unassigned columns of row i0 = argmin a and
// column j0 = argmin b, (iii) turns it into a bound on the sum, and (iv) labels only the columns (i, j) with a_i and b_j
// below that bound -- every column that attains the true minimum is among them (in the enumeration of the chain row
// that gives its label), each is labelled exactly over the whole chain, and the usual (value, position) order picks
// the winner: the result is identical to the exhaustive scan.
__device__ void VirtualCost::scan_unassigned(const LsapState& st, int t, int nov, Cand& best, int nthreads, int tid) const {
    if (!transposed || wa == nullptr) {
        lsap_scan_unassigned_full(st, *this, t, nov, best, nthreads, tid);
        return;
    }
    const Scene& S = *sc;
    const int lane = tid & 31, w = tid >> 5, nw = (nthreads + 31) >> 5;
    const int N = S.N, M = S.M, D = S.Dmax;
    double* sa = wa + (size_t)w * D;
    double* sb = wb + (size_t)w * D;
    short* il = wil + (size_t)w * D;
    short* jl = wjl + (size_t)w * D;
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    for (int a = w; a <= t; a += nw) {
        const int k = st.crow[a];
        const double cm = st.cm[a], cu = st.cu[a];
        double amin = INF, bmin = INF;
        int i0 = 0x7fffffff, j0 = 0x7fffffff;
        for (int i = lane; i < N; i += 32) {
            const double v = S.e13(i, k);
            sa[i] = v;
            if (v < amin) { amin = v; i0 = i; }
        }
        for (int j = lane; j < M; j += 32) {
            const double v = S.e23(j, k);
            sb[j] = v;
            if (v < bmin) { bmin = v; j0 = j; }
        }
        const double wamin = warp_min_d(amin), wbmin = warp_min_d(bmin);
        i0 = warp_min_i(amin == wamin ? i0 : 0x7fffffff);
        j0 = warp_min_i(bmin == wbmin ? j0 : 0x7fffffff);
        if (i0 >= N) i0 = 0;
        if (j0 >= M) j0 = 0;
        __syncwarp();
        // upper bound on the lowest label: any unassigned column's r_a
        double rub = INF;
        for (int j = lane; j < M; j += 32)
            if (!st.assigned(i0 * M + j))
                rub = fmin(rub, dsub(dadd(cm, (double)cost_from_sum(dadd(dadd(S.e12(i0, j), sa[i0]), sb[j]))), cu));
        for (int i = lane; i < N; i += 32)
            if (!st.assigned(i * M + j0))
                rub = fmin(rub, dsub(dadd(cm, (double)cost_from_sum(dadd(dadd(S.e12(i, j0), sa[i]), sb[j0]))), cu));
        rub = warp_min_d(rub);
        // r_a(c) <= rub  =>  c <= (rub + cu - cm) up to rounding of the two additions  =>  sum <= 3 c (1 + 2^-23)
        double sbound = INF;
        if (rub < INF) {
            const double cb = dadd(dadd(dsub(rub, cm), cu), dmul(1e-9, dadd(dadd(fabs(rub), fabs(cm)), dadd(fabs(cu), 1.0))));
            sbound = dadd(dmul(dmul(3.0, cb), 1.0 + 2.384185791015625e-07), 1e-30);
        }
        int nI = 0, nJ = 0;
        for (int base = 0; base < N; base += 32) {
            const int i = base + lane;
            const bool p = i < N && sa[i] <= sbound;
            const unsigned m = __ballot_sync(0xffffffffu, p);
            if (p) il[nI + __popc(m & ((1u << lane) - 1))] = (short)i;
            nI += __popc(m);
        }
        for (int base = 0; base < M; base += 32) {
            const int j = base + lane;
            const bool p = j < M && sb[j] <= sbound;
            const unsigned m = __ballot_sync(0xffffffffu, p);
            if (p) jl[nJ + __popc(m & ((1u << lane) - 1))] = (short)j;
            nJ += __popc(m);
        }
        __syncwarp();
        const int npair = nI * nJ;
        double lub = rub;                                      // tightens as this lane finds candidates
        for (int q = lane; q < npair; q += 32) {
            const int ii = q / nJ, jj = q - ii * nJ;
            const int i = il[ii], j = jl[jj];
            const int col = i * M + j;
            if (st.assigned(col)) continue;
            const double ra = dsub(dadd(cm, (double)cost_from_sum(dadd(dadd(S.e12(i, j), sa[i]), sb[j]))), cu);
            if (ra > lub) continue;                            // cannot be (or tie) the minimum
            const Cand c = lsap_label(st, *this, col, t, nov);
            if (cand_better(c, best)) best = c;
            lub = fmin(lub, c.val);
        }
        __syncwarp();                                          // the scratch is reused by this warp's next chain row
    }
}

// ------------------------------------------------------------------------------------------------------
// NaN test of a scene's virtual cost tensor (only for scenes whose scene_load reported a suspect input)
// ------------------------------------------------------------------------------------------------------
// An entry is NaN iff one of its three pair distances is (they are >= 0 or NaN), so every pair of the three pair
// matrices is tested, O(N*M + N*P + M*P) < 2^24 pairs (Dmax <= 2048).
__device__ __forceinline__ int scene_has_nan_cost(const Scene& sc, int nthreads, int tid) {
    const int M = sc.M, P = sc.P, nNM = sc.N * M, nNP = sc.N * P, nMP = M * P;
    int nan = 0;
    for (int e = tid; e < nNM + nNP + nMP; e += nthreads) {
        double d;
        if (e < nNM) d = sc.e12(e / M, e % M);
        else if (e < nNM + nNP) d = sc.e13((e - nNM) / P, (e - nNM) % P);
        else d = sc.e23((e - nNM - nNP) / P, (e - nNM - nNP) % P);
        nan |= d != d;
    }
    return nan;
}

// ------------------------------------------------------------------------------------------------------
// shared-memory layout of bpc_match_kernel
// ------------------------------------------------------------------------------------------------------
struct MatchSmem {
    double* F;       // [3][9]
    double* Pm;      // [3][12]
    Scene sc;
    LsapState st;
    RowMin rm;
    float* mcost;    // [Dmax] per assigned row
    int* mr;         // [Dmax]
    int* mk;         // [Dmax]
    double* wa;      // [nwarps][Dmax]
    double* wb;      // [nwarps][Dmax]
    short* wil;      // [nwarps][Dmax]
    short* wjl;      // [nwarps][Dmax]
};

static size_t match_smem_bytes(int Dmax, int nwarps) {
    size_t b = 0;
    b += (27 + 36) * 8;
    b += (size_t)3 * Dmax * 2 * 8;                  // pts
    b += (size_t)6 * Dmax * 3 * 8;                  // lines
    b += (size_t)nwarps * Dmax * 8 * 2;             // wa, wb
    b += lsap_state_bytes(Dmax, Dmax * Dmax);
    b += (size_t)Dmax * 4 * 6;                      // rm.cmin, rlo, cnt, mcost, mr, mk
    b += (size_t)nwarps * Dmax * 2 * 2;             // wil, wjl
    b += (size_t)6 * Dmax;                          // lvalid
    return (b + 64 + 15) & ~(size_t)15;
}

__device__ void match_carve(MatchSmem& ms, unsigned char* p, int Dmax, int nwarps) {
    ms.F = (double*)p; p += 27 * 8;
    ms.Pm = (double*)p; p += 36 * 8;
    ms.sc.pts = (double*)p; p += (size_t)3 * Dmax * 2 * 8;
    ms.sc.lines = (double*)p; p += (size_t)6 * Dmax * 3 * 8;
    ms.wa = (double*)p; p += (size_t)nwarps * Dmax * 8;
    ms.wb = (double*)p; p += (size_t)nwarps * Dmax * 8;
    p = lsap_state_carve(ms.st, p, Dmax, Dmax * Dmax);
    ms.rm.cmin = (float*)p; p += (size_t)Dmax * 4;
    ms.rm.rlo = (int*)p; p += (size_t)Dmax * 4;
    ms.rm.cnt = (int*)p; p += (size_t)Dmax * 4;
    ms.mcost = (float*)p; p += (size_t)Dmax * 4;
    ms.mr = (int*)p; p += (size_t)Dmax * 4;
    ms.mk = (int*)p; p += (size_t)Dmax * 4;
    ms.wil = (short*)p; p += (size_t)nwarps * Dmax * 2;
    ms.wjl = (short*)p; p += (size_t)nwarps * Dmax * 2;
    ms.sc.lvalid = (uint8_t*)p;
    ms.sc.Dmax = Dmax;
}

// ------------------------------------------------------------------------------------------------------
// PoseEstimator._match for one scene per CTA
// ------------------------------------------------------------------------------------------------------
// SPILL = false: the scene's state is carved out of shared memory (the compiler then addresses it with LDS / STS, not generic
// loads); SPILL = true: a per-CTA block of the caller's workspace (Dmax beyond ~550)
template <bool SPILL>
__global__ void __launch_bounds__(256, 2) bpc_match_kernel(const float* __restrict__ Ks, const double* __restrict__ RTs,
                                 const double* __restrict__ centers, const int32_t* __restrict__ counts,
                                 int S, int Dmax, float threshold,
                                 int32_t* __restrict__ idx, int32_t* __restrict__ nout, float* __restrict__ costout,
                                 double* __restrict__ Xout, double* __restrict__ reproj, double* __restrict__ Fout,
                                 unsigned char* __restrict__ spill, size_t spill_per_cta) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, nth = blockDim.x, nwarps = nth >> 5;
    MatchSmem ms;
    // scenes too large for shared memory (Dmax > ~450) keep their state in the caller's workspace, one block per CTA
    if (SPILL) match_carve(ms, spill + (size_t)blockIdx.x * spill_per_cta, Dmax, nwarps);
    else match_carve(ms, smem_raw, Dmax, nwarps);
    const double NaN = __longlong_as_double(0x7ff8000000000000LL);

    for (int s = blockIdx.x; s < S; s += gridDim.x) {
        __syncthreads();                                   // previous scene fully written out
        Scene& sc = ms.sc;
        sc.N = counts[s * 3 + 0]; sc.M = counts[s * 3 + 1]; sc.P = counts[s * 3 + 2];
        sc.m_magic = sc.M > 0 ? (1ull << 40) / (unsigned long long)sc.M + 1ull : 0ull;
        const float* K = Ks + (size_t)s * 27;
        const double* RT = RTs + (size_t)s * 48;
        // ---- phase 0 ---------------------------------------------------------------------------------
        if (tid < 3) {
            const int a = (tid == 2) ? 1 : 0, b = (tid == 0) ? 1 : 2;        // pairs 12, 13, 23
            fundamental(K + a * 9, RT + a * 16, K + b * 9, RT + b * 16, ms.F + tid * 9);
        }
        __syncthreads();
        if (Fout != nullptr && tid < 27) Fout[(size_t)s * 27 + tid] = ms.F[tid];
        const int N = sc.N, M = sc.M, P = sc.P;
        // padding of the outputs
        for (int e = tid; e < Dmax; e += nth) {
            idx[((size_t)s * Dmax + e) * 3 + 0] = -1; idx[((size_t)s * Dmax + e) * 3 + 1] = -1; idx[((size_t)s * Dmax + e) * 3 + 2] = -1;
            costout[(size_t)s * Dmax + e] = __int_as_float(0x7fc00000);
            for (int c = 0; c < 3; ++c) {
                Xout[((size_t)s * Dmax + e) * 3 + c] = NaN;
                if (reproj != nullptr) reproj[((size_t)s * Dmax + e) * 3 + c] = NaN;
            }
        }
        if (N > Dmax || M > Dmax || P > Dmax) {              // e.g. the overflow count of bpc_detections_from_yolo
            if (tid == 0) nout[s] = BPC_N_OVERFLOW;
            continue;
        }
        if (N <= 0 || M <= 0 || P <= 0) {                    // process_pose.py:161-163
            if (tid == 0) nout[s] = 0;
            continue;
        }
        const bool suspect = scene_load(sc, ms.F, centers + (size_t)s * 3 * Dmax * 2, nth, tid);
        const int NM = N * M;
        const int transposed = NM > P;                       // SciPy: transpose iff more rows than columns
        const int nr = transposed ? P : NM, nc = transposed ? NM : P;
        lsap_reset(ms.st, nr, nc, nth, tid);
        // a non-finite (or huge) centre or line: SciPy rejects the cost tensor if any entry is NaN (BPC_N_INFEASIBLE)
        if (__syncthreads_or(suspect) && __syncthreads_or(scene_has_nan_cost(sc, nth, tid))) {
            if (tid == 0) nout[s] = BPC_N_INFEASIBLE;
            continue;
        }
        // ---- phase 1 ---------------------------------------------------------------------------------
        if (transposed) {
            const int w = warp_id();
            for (int k = w; k < P; k += nwarps)
                row_argmin(sc, k, ms.wa + (size_t)w * Dmax, ms.wb + (size_t)w * Dmax,
                           ms.wil + (size_t)w * Dmax, ms.wjl + (size_t)w * Dmax, ms.rm);
        }
        __syncthreads();
        // ---- phase 2 ---------------------------------------------------------------------------------
        VirtualCost acc;
        acc.sc = &sc; acc.transposed = transposed;
        acc.wa = ms.wa; acc.wb = ms.wb; acc.wil = ms.wil; acc.wjl = ms.wjl;
        LsapState& st = ms.st;
        int row = 0;
        for (;;) {
            if (tid == 0) {
                int r = row;
                if (transposed) {
                    // an unassigned unique argmin column is an immediate sink: every other column has a
                    // strictly larger cost and v <= 0, so its reduced cost is strictly larger
                    while (r < nr && ms.rm.cnt[r] == 1 && !st.assigned(ms.rm.rlo[r])) {
                        const int col = ms.rm.rlo[r];
                        st.col4row[r] = col; st.vcol[r] = 0.0; st.set_assigned(col);
                        st.u[r] = (double)ms.rm.cmin[r];
                        ++r;
                    }
                }
                st.ctl[0] = r;
            }
            __syncthreads();
            row = st.ctl[0];
            if (row >= nr) break;
            lsap_augment(st, acc, row, nth, tid);
            if (st.ctl[2]) break;
            ++row;
        }
        __syncthreads();
        if (st.ctl[2]) {                                     // infeasible (a row of +inf costs): SciPy raises
            if (tid == 0) nout[s] = BPC_N_INFEASIBLE;
            continue;
        }
        // ---- phase 3 ---------------------------------------------------------------------------------
        for (int rrow = tid; rrow < nr; rrow += nth) {
            const int col = st.col4row[rrow];
            const int r = transposed ? col : rrow, k = transposed ? rrow : col;
            const int i = r / M, j = r - i * M;
            const float c = sc.cost(i, j, k);
            ms.mcost[rrow] = c; ms.mr[rrow] = (c < threshold) ? r : -1; ms.mk[rrow] = k;
        }
        __syncthreads();
        int kept = 0;
        for (int e = 0; e < nr; ++e) kept += (ms.mr[e] >= 0);
        if (tid == 0) nout[s] = kept;
        for (int rrow = tid; rrow < nr; rrow += nth) {
            const int r = ms.mr[rrow];
            if (r < 0) continue;
            const float c = ms.mcost[rrow];
            int rank = 0;
            for (int e = 0; e < nr; ++e) {
                const int re = ms.mr[e];
                if (re < 0) continue;
                const float ce = ms.mcost[e];
                rank += (ce < c) || (ce == c && re < r);
            }
            const int k = ms.mk[rrow];
            const int i = r / M, j = r - i * M;
            const size_t o = (size_t)s * Dmax + rank;
            idx[o * 3 + 0] = i; idx[o * 3 + 1] = j; idx[o * 3 + 2] = k;
            costout[o] = c;                  // triangulation of the match: bpc_match_tri_kernel (register budget)
        }
    }
}

// DLT triangulation + reprojection error of every match written by bpc_match_kernel, one thread per match slot.
// (A separate launch keeps the 80 live doubles of the Jacobi sweep out of the matcher's register allocation.)
__global__ void __launch_bounds__(128)
bpc_match_tri_kernel(const float* __restrict__ Ks, const double* __restrict__ RTs, const double* __restrict__ centers,
                     const int32_t* __restrict__ idx, const int32_t* __restrict__ n, int S, int Dmax,
                     double* __restrict__ Xout, double* __restrict__ reproj) {
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t >= (long long)S * Dmax) return;
    const int s = (int)(t / Dmax), slot = (int)(t - (long long)s * Dmax);
    if (slot >= n[s]) return;
    double Pm[36], xy[6], X[3];
    for (int c = 0; c < 3; ++c) {
        projection(Ks + (size_t)s * 27 + c * 9, RTs + (size_t)s * 48 + c * 16, Pm + c * 12);
        const int d = idx[(size_t)t * 3 + c];
        const double* p = centers + (((size_t)s * 3 + c) * Dmax + d) * 2;
        xy[c * 2] = p[0]; xy[c * 2 + 1] = p[1];
    }
    triangulate3(Pm, xy, X);
    Xout[(size_t)t * 3 + 0] = X[0]; Xout[(size_t)t * 3 + 1] = X[1]; Xout[(size_t)t * 3 + 2] = X[2];
    if (reproj != nullptr)
        for (int v = 0; v < 3; ++v) reproj[(size_t)t * 3 + v] = reprojection(Pm + v * 12, X, xy + v * 2);
}

// ------------------------------------------------------------------------------------------------------
// match_objects on an explicit cost tensor (epipolar_matching.py:100-116), one CTA per problem
// ------------------------------------------------------------------------------------------------------
__global__ void bpc_match_objects_kernel(const float* __restrict__ cost, int S, int N, int M, int P, float threshold,
                                         int32_t* __restrict__ idx, int32_t* __restrict__ nout) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, nth = blockDim.x;
    const int NM = N * M;
    const int transposed = NM > P;
    const int nr = transposed ? P : NM, nc = transposed ? NM : P;
    LsapState st;
    unsigned char* p = lsap_state_carve(st, smem_raw, nr, nc);
    int* keep = (int*)p;                                    // [nr]
    for (int s = blockIdx.x; s < S; s += gridDim.x) {
        __syncthreads();
        lsap_reset(st, nr, nc, nth, tid);
        __syncthreads();
        ExplicitCost acc;
        acc.c = cost + (size_t)s * NM * P; acc.P = P; acc.transposed = transposed;
        // SciPy rejects a matrix with ANY NaN or -inf entry ("matrix contains invalid numeric entries")
        int invalid = 0;
        for (long long e = tid; e < (long long)NM * P; e += nth) {
            const float v = acc.c[e];
            invalid |= (v != v) || (v == __int_as_float(0xff800000));
        }
        bool bad = __syncthreads_or(invalid) != 0;
        for (int row = 0; row < nr && !bad; ++row) {
            lsap_augment(st, acc, row, nth, tid);
            if (st.ctl[2]) { bad = true; break; }
        }
        __syncthreads();
        for (int e = tid; e < nr; e += nth) {
            idx[((size_t)s * nr + e) * 3 + 0] = -1; idx[((size_t)s * nr + e) * 3 + 1] = -1; idx[((size_t)s * nr + e) * 3 + 2] = -1;
        }
        if (bad) {
            if (tid == 0) nout[s] = -1;
            continue;
        }
        for (int rrow = tid; rrow < nr; rrow += nth) {
            const int col = st.col4row[rrow];
            const int r = transposed ? col : rrow, k = transposed ? rrow : col;
            keep[rrow] = (acc.c[(size_t)r * P + k] < threshold) ? r : -1;
        }
        __syncthreads();
        int kept = 0;
        for (int e = 0; e < nr; ++e) kept += (keep[e] >= 0);
        if (tid == 0) nout[s] = kept;
        for (int rrow = tid; rrow < nr; rrow += nth) {
            const int r = keep[rrow];
            if (r < 0) continue;
            int rank = 0;                                    // ascending r (SciPy's output order)
            for (int e = 0; e < nr; ++e) rank += (keep[e] >= 0 && keep[e] < r);
            const int k = transposed ? rrow : st.col4row[rrow];
            const size_t o = (size_t)s * nr + rank;
            idx[o * 3 + 0] = r / M; idx[o * 3 + 1] = r % M; idx[o * 3 + 2] = k;
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// small stand-alone kernels
// ------------------------------------------------------------------------------------------------------
__global__ void bpc_fundamental_kernel(const float* __restrict__ Ks, const double* __restrict__ RTs, int S, double* __restrict__ F) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= S * 3) return;
    const int s = t / 3, pr = t - s * 3;
    const int a = (pr == 2) ? 1 : 0, b = (pr == 0) ? 1 : 2;
    double f[9];
    fundamental(Ks + (size_t)s * 27 + a * 9, RTs + (size_t)s * 48 + a * 16, Ks + (size_t)s * 27 + b * 9,
                RTs + (size_t)s * 48 + b * 16, f);
    for (int e = 0; e < 9; ++e) F[(size_t)t * 9 + e] = f[e];
}

__global__ void bpc_cost_tensor_kernel(const double* __restrict__ F, const double* __restrict__ centers,
                                       const int32_t* __restrict__ counts, int S, int Dmax, float* __restrict__ cost) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, nth = blockDim.x;
    double* Fs = (double*)smem_raw;
    Scene sc;
    sc.pts = Fs + 27 + 1;
    sc.lines = sc.pts + (size_t)3 * Dmax * 2;
    sc.lvalid = (uint8_t*)(sc.lines + (size_t)6 * Dmax * 3);
    sc.Dmax = Dmax;
    for (int s = blockIdx.x; s < S; s += gridDim.x) {
        __syncthreads();
        if (tid < 27) Fs[tid] = F[(size_t)s * 27 + tid];
        sc.N = counts[s * 3 + 0]; sc.M = counts[s * 3 + 1]; sc.P = counts[s * 3 + 2];
        sc.m_magic = sc.M > 0 ? (1ull << 40) / (unsigned long long)sc.M + 1ull : 0ull;
        __syncthreads();
        if (sc.N < 0 || sc.M < 0 || sc.P < 0 || sc.N > Dmax || sc.M > Dmax || sc.P > Dmax) continue;
        scene_load(sc, Fs, centers + (size_t)s * 3 * Dmax * 2, nth, tid);
        __syncthreads();
        const int N = sc.N, M = sc.M, P = sc.P;
        const long long total = (long long)N * M * P;
        for (long long e = tid; e < total; e += nth) {
            const int k = (int)(e % P);
            const int r = (int)(e / P);
            const int i = r / M, j = r - i * M;
            cost[(((size_t)s * Dmax + i) * Dmax + j) * Dmax + k] = sc.cost(i, j, k);
        }
    }
}

// P = K (float32) @ RT[:3] (float64) for n cameras (process_pose.py:91)
__global__ void bpc_projection_kernel(const float* __restrict__ K, const double* __restrict__ RT, int n, double* __restrict__ P) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    double pm[12];
    projection(K + (size_t)t * 9, RT + (size_t)t * 16, pm);
    for (int e = 0; e < 12; ++e) P[(size_t)t * 12 + e] = pm[e];
}

__global__ void bpc_triangulate_kernel(const double* __restrict__ P, const double* __restrict__ pts, int n, double* __restrict__ X) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    double Pm[36], xy[6], x[3];
    for (int e = 0; e < 36; ++e) Pm[e] = P[(size_t)t * 36 + e];
    for (int e = 0; e < 6; ++e) xy[e] = pts[(size_t)t * 6 + e];
    triangulate3(Pm, xy, x);
    X[(size_t)t * 3 + 0] = x[0]; X[(size_t)t * 3 + 1] = x[1]; X[(size_t)t * 3 + 2] = x[2];
}

// epipolar_error(pt1, pt2, F) for n independent (pt1, pt2, F) triples (epipolar_matching.py:5-28)
__global__ void bpc_epipolar_error_kernel(const double* __restrict__ F, const double* __restrict__ p1, const double* __restrict__ p2,
                                          int n, double* __restrict__ e) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    double f[9], l1[3], l2[3];
    for (int k = 0; k < 9; ++k) f[k] = F[(size_t)t * 9 + k];
    const double x1 = p1[(size_t)t * 2], y1 = p1[(size_t)t * 2 + 1], x2 = p2[(size_t)t * 2], y2 = p2[(size_t)t * 2 + 1];
    const bool ok2 = epiline(f, 0, x1, y1, l2);       // l2 = F @ pt1: line in the second camera
    const bool ok1 = epiline(f, 1, x2, y2, l1);       // l1 = F.T @ pt2
    const double d1 = ok1 ? line_point(l1, x1, y1) : 9999.0;
    const double d2 = ok2 ? line_point(l2, x2, y2) : 9999.0;
    e[t] = dmul(0.5, dadd(d1, d2));
}

// epipolar_error_full(pt1, pt2, pt3, F12, F13, F23) for n triples (epipolar_matching.py:73-81); F = [n][3][9]
__global__ void bpc_epipolar_error_full_kernel(const double* __restrict__ F, const double* __restrict__ pts, int n, double* __restrict__ e) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const double* p = pts + (size_t)t * 6;
    double acc[3];
    const int ia[3] = {0, 0, 1}, ib[3] = {1, 2, 2};
    for (int pr = 0; pr < 3; ++pr) {
        double f[9], l1[3], l2[3];
        for (int k = 0; k < 9; ++k) f[k] = F[((size_t)t * 3 + pr) * 9 + k];
        const double xa = p[ia[pr] * 2], ya = p[ia[pr] * 2 + 1], xb = p[ib[pr] * 2], yb = p[ib[pr] * 2 + 1];
        const bool ok2 = epiline(f, 0, xa, ya, l2);
        const bool ok1 = epiline(f, 1, xb, yb, l1);
        const double d1 = ok1 ? line_point(l1, xa, ya) : 9999.0;
        const double d2 = ok2 ? line_point(l2, xb, yb) : 9999.0;
        acc[pr] = dmul(0.5, dadd(d1, d2));
    }
    e[t] = ddiv(dadd(dadd(acc[0], acc[1]), acc[2]), 3.0);
}

// DLT for V views (2 <= V <= 8), one thread per point; same one-sided Jacobi as triangulate3 on a (2V x 4) matrix
__global__ void bpc_triangulate_views_kernel(const double* __restrict__ P, const double* __restrict__ pts, int n, int V, double* __restrict__ X) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    double A[16][4], Vm[4][4];
    const int rows = 2 * V;
    for (int v = 0; v < V; ++v) {
        const double* Pm = P + ((size_t)t * V + v) * 12;
        const double x = pts[((size_t)t * V + v) * 2], y = pts[((size_t)t * V + v) * 2 + 1];
        for (int c = 0; c < 4; ++c) {
            A[2 * v][c] = dsub(dmul(x, Pm[8 + c]), Pm[c]);
            A[2 * v + 1][c] = dsub(dmul(y, Pm[8 + c]), Pm[4 + c]);
        }
    }
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) Vm[r][c] = (r == c) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 20; ++sweep) {
        bool rotated = false;
        for (int p = 0; p < 3; ++p)
            for (int q = p + 1; q < 4; ++q) {
                double alpha = 0.0, beta = 0.0, gamma = 0.0;
                for (int r = 0; r < rows; ++r) { alpha += A[r][p] * A[r][p]; beta += A[r][q] * A[r][q]; gamma += A[r][p] * A[r][q]; }
                if (fabs(gamma) > 1e-15 * sqrt(alpha * beta) && fabs(gamma) > 1e-300) {
                    const double zeta = (beta - alpha) / (2.0 * gamma);
                    const double tt = fabs(zeta) > 1e150 ? 0.5 / zeta : copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                    const double cs = 1.0 / sqrt(1.0 + tt * tt), sn = cs * tt;
                    for (int r = 0; r < rows; ++r) { const double ap = A[r][p], aq = A[r][q]; A[r][p] = cs * ap - sn * aq; A[r][q] = sn * ap + cs * aq; }
                    for (int r = 0; r < 4; ++r) { const double vp = Vm[r][p], vq = Vm[r][q]; Vm[r][p] = cs * vp - sn * vq; Vm[r][q] = sn * vp + cs * vq; }
                    rotated = true;
                }
            }
        if (!rotated) break;
    }
    double best = 0.0; int bi = 0;
    for (int c = 0; c < 4; ++c) {
        double nrm = 0.0;
        for (int r = 0; r < rows; ++r) nrm += A[r][c] * A[r][c];
        if (c == 0 || nrm < best) { best = nrm; bi = c; }
    }
    X[(size_t)t * 3 + 0] = Vm[0][bi] / Vm[3][bi];
    X[(size_t)t * 3 + 1] = Vm[1][bi] / Vm[3][bi];
    X[(size_t)t * 3 + 2] = Vm[2][bi] / Vm[3][bi];
}

__global__ void bpc_reproj_kernel(const double* __restrict__ P, const double* __restrict__ X, const double* __restrict__ pts,
                                  int n, double* __restrict__ err) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * 3) return;
    const int m = t / 3;
    double Pm[12];
    for (int e = 0; e < 12; ++e) Pm[e] = P[(size_t)t * 12 + e];
    err[t] = reprojection(Pm, X + (size_t)m * 3, pts + (size_t)t * 2);
}

// Detector post-processing (process_pose.py:123-141): keep class 0 with conf >= threshold, int() every box
// coordinate (truncation toward zero), centre = 0.5 * (x1 + x2); order preserved.  One warp per (scene, camera).
__global__ void bpc_detections_kernel(const float* __restrict__ xyxy, const float* __restrict__ conf, const float* __restrict__ cls,
                                      const int32_t* __restrict__ nraw, int SC, int Nraw, float thresh, int Dmax,
                                      int32_t* __restrict__ boxes, double* __restrict__ centers, int32_t* __restrict__ counts) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= SC) return;
    const int n = min(max(nraw[w], 0), Nraw);
    int kept = 0;
    for (int base = 0; base < n; base += 32) {
        const int d = base + lane;
        bool keep = false;
        if (d < n) keep = (cls[(size_t)w * Nraw + d] == 0.f) && (conf[(size_t)w * Nraw + d] >= thresh);
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        const int pos = kept + __popc(m & ((1u << lane) - 1));
        if (keep && pos < Dmax) {
            const float4 b = reinterpret_cast<const float4*>(xyxy)[(size_t)w * Nraw + d];
            const int x1 = __float2int_rz(b.x), y1 = __float2int_rz(b.y), x2 = __float2int_rz(b.z), y2 = __float2int_rz(b.w);
            reinterpret_cast<int4*>(boxes)[(size_t)w * Dmax + pos] = make_int4(x1, y1, x2, y2);
            centers[((size_t)w * Dmax + pos) * 2 + 0] = 0.5 * (double)((long long)x1 + x2);
            centers[((size_t)w * Dmax + pos) * 2 + 1] = 0.5 * (double)((long long)y1 + y2);
        }
        kept += __popc(m);
    }
    if (lane == 0) counts[w] = kept;          // may exceed Dmax: the caller sees the overflow
}

__global__ void bpc_box_centers_kernel(const int32_t* __restrict__ boxes, int count, double* __restrict__ centers) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const int4 b = reinterpret_cast<const int4*>(boxes)[t];
    // 0.5 * (x1 + x2) on Python ints (process_pose.py:135-136): the integer sum is exact
    centers[(size_t)t * 2 + 0] = 0.5 * (double)((long long)b.x + (long long)b.z);
    centers[(size_t)t * 2 + 1] = 0.5 * (double)((long long)b.y + (long long)b.w);
}

// Optional reprojection-error filter (the helper compute_reprojection_error, utils/triangulation.py:14-18, has no caller in
// the reference, so the policy is this library's: a match is dropped when ANY view's error exceeds the threshold; the
// survivors keep their (cost, r) order).  One thread per scene, in place; the tail is re-padded.
__global__ void bpc_match_filter_kernel(int S, int Dmax, double thresh, int32_t* __restrict__ idx, int32_t* __restrict__ n,
                                        float* __restrict__ cost, double* __restrict__ X, double* __restrict__ reproj) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int cnt = n[s];
    if (cnt <= 0) return;
    const double NaN = __longlong_as_double(0x7ff8000000000000LL);
    const size_t base = (size_t)s * Dmax;
    int kept = 0;
    for (int m = 0; m < cnt; ++m) {
        const double* e = reproj + (base + m) * 3;
        if (e[0] > thresh || e[1] > thresh || e[2] > thresh) continue;
        if (kept != m) {
            for (int c = 0; c < 3; ++c) {
                idx[(base + kept) * 3 + c] = idx[(base + m) * 3 + c];
                X[(base + kept) * 3 + c] = X[(base + m) * 3 + c];
                reproj[(base + kept) * 3 + c] = e[c];
            }
            cost[base + kept] = cost[base + m];
        }
        ++kept;
    }
    for (int m = kept; m < cnt; ++m) {
        for (int c = 0; c < 3; ++c) { idx[(base + m) * 3 + c] = -1; X[(base + m) * 3 + c] = NaN; reproj[(base + m) * 3 + c] = NaN; }
        cost[base + m] = __int_as_float(0x7fc00000);
    }
    n[s] = kept;
}

// Pose records for the final gather (SURVEY.md 8e): the valid match slots of every scene, compacted in scene order, as
// 64-byte records (idx i32 x3, cost f32, X f64 x3, reproj f64 x3), behind a header and the per-scene counts.
//   buffer = | total i32, S i32, Kmax i32, 0 | n[S] i32 (padded to 16 bytes) | records ...
struct __align__(16) PoseRecord { int32_t i, j, k; float cost; double X[3]; double reproj[3]; };
static_assert(sizeof(PoseRecord) == 64, "PoseRecord layout");
__host__ __device__ inline size_t pack_records_offset(int S) { return 16 + (((size_t)S * 4 + 15) & ~(size_t)15); }

__global__ void bpc_pack_records_kernel(const int32_t* __restrict__ idx, const int32_t* __restrict__ n, const float* __restrict__ cost,
                                        const double* __restrict__ X, const double* __restrict__ reproj,
                                        const int32_t* __restrict__ scene_offset, int offset_div, int S, int Kmax,
                                        unsigned char* __restrict__ buf) {
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    int32_t* head = reinterpret_cast<int32_t*>(buf);
    if (t == 0) { head[0] = scene_offset[S] / offset_div; head[1] = S; head[2] = Kmax; head[3] = 0; }
    if (t < S) head[4 + t] = n[t];
    else if (t < ((S + 3) & ~3)) head[4 + t] = 0;             // padding of the counts up to the 16-byte record base
    if (t >= (long long)S * Kmax) return;
    const int s = (int)(t / Kmax), m = (int)(t - (long long)s * Kmax);
    if (m >= n[s]) return;
    PoseRecord r;
    r.i = idx[t * 3]; r.j = idx[t * 3 + 1]; r.k = idx[t * 3 + 2];
    r.cost = cost[t];
    const double NaN = __longlong_as_double(0x7ff8000000000000LL);
    for (int c = 0; c < 3; ++c) { r.X[c] = X[t * 3 + c]; r.reproj[c] = reproj ? reproj[t * 3 + c] : NaN; }
    PoseRecord* out = reinterpret_cast<PoseRecord*>(buf + pack_records_offset(S)) + (scene_offset[s] / offset_div + m);
    const uint4* src = reinterpret_cast<const uint4*>(&r);
    uint4* dst = reinterpret_cast<uint4*>(out);
    dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2]; dst[3] = src[3];
}

// ROI records: single CTA exclusive scan over 3*n[s], then a grid-stride fill.
__global__ void bpc_roi_offsets_kernel(const int32_t* __restrict__ n, int S, int32_t* __restrict__ offs) {
    __shared__ int part[1024];
    const int tid = threadIdx.x, nth = blockDim.x;
    const int per = (S + nth - 1) / nth;
    const int lo = min(S, tid * per), hi = min(S, lo + per);
    int sum = 0;
    for (int s = lo; s < hi; ++s) sum += 3 * max(0, n[s]);
    part[tid] = sum;
    __syncthreads();
    if (tid == 0) {
        int acc = 0;
        for (int t = 0; t < nth; ++t) { const int v = part[t]; part[t] = acc; acc += v; }
        offs[S] = acc;
    }
    __syncthreads();
    int acc = part[tid];
    for (int s = lo; s < hi; ++s) { offs[s] = acc; acc += 3 * max(0, n[s]); }
}

__global__ void bpc_roi_fill_kernel(const int32_t* __restrict__ boxes, const int32_t* __restrict__ idx, const int32_t* __restrict__ n,
                                    const int32_t* __restrict__ image_of_scene, int S, int Dmax, int Kmax,
                                    const int32_t* __restrict__ offs, int32_t* __restrict__ rois) {
    const long long total = (long long)S * Kmax * 3;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int v = (int)(e % 3);
        const int m = (int)((e / 3) % Kmax);
        const int s = (int)(e / (3LL * Kmax));
        if (m >= n[s]) continue;
        const int d = idx[((size_t)s * Kmax + m) * 3 + v];
        const int32_t* b = boxes + (((size_t)s * 3 + v) * Dmax + d) * 4;
        int32_t* o = rois + ((size_t)offs[s] + (size_t)m * 3 + v) * 5;
        o[0] = image_of_scene[s * 3 + v]; o[1] = b[0]; o[2] = b[1]; o[3] = b[2]; o[4] = b[3];
    }
}

// ------------------------------------------------------------------------------------------------------
// host launchers (C ABI)
// ------------------------------------------------------------------------------------------------------
constexpr size_t MATCH_MAX_SMEM = 227 * 1024;

static int pick_threads(int Dmax) {
    if (Dmax <= 32) return 32;
    if (Dmax <= 64) return 128;
    return 256;
}

}  // namespace bpc

using namespace bpc;

extern "C" int bpc_fundamental(const float* Ks, const double* RTs, int S, double* F, void* stream) {
    if (S < 0 || (S > 0 && (!Ks || !RTs || !F))) return BPC_EINVAL;
    if (S == 0) return BPC_OK;
    bpc_fundamental_kernel<<<(S * 3 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(Ks, RTs, S, F);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

extern "C" int bpc_cost_tensor(const double* F, const double* centers, const int32_t* counts, int S, int Dmax,
                               float* cost, void* stream) {
    if (S < 0 || Dmax < 1 || (S > 0 && (!F || !centers || !counts || !cost))) return BPC_EINVAL;
    if (Dmax > BPC_MAX_DET) return BPC_ETOOBIG;
    if (S == 0) return BPC_OK;
    const size_t smem = (28 + (size_t)3 * Dmax * 2 + (size_t)6 * Dmax * 3) * 8 + (size_t)6 * Dmax + 16;
    if (smem > MATCH_MAX_SMEM) return BPC_ETOOBIG;
    cudaError_t e = cudaFuncSetAttribute(bpc_cost_tensor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MATCH_MAX_SMEM);
    if (e != cudaSuccess) return (int)e;
    bpc_cost_tensor_kernel<<<S, 256, smem, (cudaStream_t)stream>>>(F, centers, counts, S, Dmax, cost);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

extern "C" int bpc_match_objects(const float* cost, int S, int N, int M, int P, float threshold,
                                 int32_t* idx, int32_t* n, void* stream) {
    if (S < 0 || N < 1 || M < 1 || P < 1 || (S > 0 && (!cost || !idx || !n))) return BPC_EINVAL;
    if ((long long)N * M > (1 << 24) || P > (1 << 24)) return BPC_ETOOBIG;
    if (S == 0) return BPC_OK;
    const int NM = N * M;
    const int nr = NM > P ? P : NM, nc = NM > P ? NM : P;
    const size_t smem = lsap_state_bytes(nr, nc) + (size_t)nr * 4 + 32;
    if (smem > MATCH_MAX_SMEM) return BPC_ETOOBIG;
    // always the same constant: idempotent, so concurrent callers cannot interleave set(small) / launch(large)
    cudaError_t e = cudaFuncSetAttribute(bpc_match_objects_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MATCH_MAX_SMEM);
    if (e != cudaSuccess) return (int)e;
    const int threads = nc <= 1024 ? 32 : (nc <= 8192 ? 128 : 256);
    bpc_match_objects_kernel<<<S, threads, smem, (cudaStream_t)stream>>>(cost, S, N, M, P, threshold, idx, n);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

// launch geometry of bpc_match_kernel for a given Dmax: threads, dynamic shared memory, and -- when even one warp's state
// does not fit the 227 KB of an SM -- the per-CTA spill block in the caller's workspace
static void match_plan(int Dmax, int* threads, size_t* smem, size_t* spill_per_cta) {
    int th = pick_threads(Dmax);
    size_t sm = match_smem_bytes(Dmax, th / 32);
    while (sm > MATCH_MAX_SMEM && th > 32) { th /= 2; sm = match_smem_bytes(Dmax, th / 32); }
    *spill_per_cta = 0;
    if (sm > MATCH_MAX_SMEM) {
        th = 256;
        *spill_per_cta = (match_smem_bytes(Dmax, th / 32) + 255) & ~(size_t)255;
        sm = 0;
    }
    *threads = th; *smem = sm;
}
static int match_grid(int S, size_t spill_per_cta) { return spill_per_cta ? (S < 2 * 148 ? S : 2 * 148) : S; }

extern "C" size_t bpc_match_workspace_bytes(int S, int Dmax) {
    if (S < 1 || Dmax < 1 || Dmax > BPC_MAX_DET) return 0;
    int threads; size_t smem, spill;
    match_plan(Dmax, &threads, &smem, &spill);
    return spill * (size_t)match_grid(S, spill);
}

extern "C" int bpc_match_triangulate(const float* Ks, const double* RTs, const double* centers, const int32_t* counts,
                                     int S, int Dmax, float threshold, int has_reproj_thresh, double reproj_thresh,
                                     int32_t* idx, int32_t* n, float* cost, double* X,
                                     double* reproj, double* F, void* workspace, size_t workspace_bytes, void* stream) {
    if (S < 0 || Dmax < 1) return BPC_EINVAL;
    if (S > 0 && (!Ks || !RTs || !centers || !counts || !idx || !n || !cost || !X)) return BPC_EINVAL;
    if (has_reproj_thresh && (!reproj || !(reproj_thresh == reproj_thresh))) return BPC_EINVAL;   // the filter reads `reproj`
    if (Dmax > BPC_MAX_DET) return BPC_ETOOBIG;
    if (S == 0) return BPC_OK;
    int threads; size_t smem, spill;
    match_plan(Dmax, &threads, &smem, &spill);
    const int grid = match_grid(S, spill);
    if (spill) {
        if (!workspace || ((uintptr_t)workspace & 15) != 0) return workspace ? BPC_EALIGN : BPC_EWORKSPACE;
        if (workspace_bytes < spill * (size_t)grid) return BPC_EWORKSPACE;
    }
    auto kern = spill ? bpc_match_kernel<true> : bpc_match_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MATCH_MAX_SMEM);
    if (e != cudaSuccess) return (int)e;
    kern<<<grid, threads, smem, (cudaStream_t)stream>>>(Ks, RTs, centers, counts, S, Dmax, threshold, idx, n, cost, X, reproj, F,
                                                        spill ? (unsigned char*)workspace : nullptr, spill);
    BPC_LAUNCH_CHECK();
    const long long slots = (long long)S * Dmax;
    bpc_match_tri_kernel<<<(unsigned)((slots + 127) / 128), 128, 0, (cudaStream_t)stream>>>(Ks, RTs, centers, idx, n, S, Dmax, X, reproj);
    BPC_LAUNCH_CHECK();
    if (has_reproj_thresh) {
        bpc_match_filter_kernel<<<(S + 127) / 128, 128, 0, (cudaStream_t)stream>>>(S, Dmax, reproj_thresh, idx, n, cost, X, reproj);
        BPC_LAUNCH_CHECK();
    }
    return BPC_OK;
}

extern "C" size_t bpc_pack_records_bytes(int S, int Kmax) {
    if (S < 0 || Kmax < 0) return 0;
    return pack_records_offset(S) + (size_t)S * Kmax * sizeof(PoseRecord);
}

extern "C" int bpc_pack_records(const int32_t* idx, const int32_t* n, const float* cost, const double* X, const double* reproj,
                                const int32_t* scene_offset, int offset_div, int S, int Kmax, void* buf, void* stream) {
    if (S < 0 || Kmax < 1 || offset_div < 1) return BPC_EINVAL;
    if (S > 0 && (!idx || !n || !cost || !X || !scene_offset || !buf)) return BPC_EINVAL;
    if (((uintptr_t)buf & 15) != 0) return BPC_EALIGN;
    if (S == 0) return BPC_OK;
    const long long slots = (long long)S * Kmax;
    bpc_pack_records_kernel<<<(unsigned)((slots + 255) / 256), 256, 0, (cudaStream_t)stream>>>(idx, n, cost, X, reproj, scene_offset, offset_div,
                                                                                              S, Kmax, (unsigned char*)buf);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

extern "C" int bpc_projection(const float* K, const double* RT, int n, double* P, void* stream) {
    if (n < 0 || (n > 0 && (!K || !RT || !P))) return BPC_EINVAL;
    if (n == 0) return BPC_OK;
    bpc_projection_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(K, RT, n, P);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

extern "C" int bpc_triangulate(const double* P, const double* pts, int n, double* X, void* stream) {
    if (n < 0 || (n > 0 && (!P || !pts || !X))) return BPC_EINVAL;
    if (n == 0) return BPC_OK;
    bpc_triangulate_kernel<<<(n + 63) / 64, 64, 0, (cudaStream_t)stream>>>(P, pts, n, X);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

extern "C" int bpc_reprojection_error(const double* P, const double* X, const double* pts, int n, double* err, void* stream) {
    if (n < 0 || (n > 0 && (!P || !pts || !X || !err))) return BPC_EINVAL;
    if (n == 0) return BPC_OK;
    bpc_reproj_kernel<<<(n * 3 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(P, X, pts, n, err);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

extern "C" int bpc_epipolar_error(const double* F, const double* pt1, const double* pt2, int n, double* e, void* stream) {
    if (n < 0 || (n > 0 && (!F || !pt1 || !pt2 || !e))) return BPC_EINVAL;
    if (n == 0) return BPC_OK;
    bpc_epipolar_error_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(F, pt1, pt2, n, e);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

extern "C" int bpc_epipolar_error_full(const double* F, const double* pts, int n, double* e, void* stream) {
    if (n < 0 || (n > 0 && (!F || !pts || !e))) return BPC_EINVAL;
    if (n == 0) return BPC_OK;
    bpc_epipolar_error_full_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(F, pts, n, e);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

extern "C" int bpc_triangulate_views(const double* P, const double* pts, int n, int V, double* X, void* stream) {
    if (n < 0 || V < 2 || V > 8 || (n > 0 && (!P || !pts || !X))) return BPC_EINVAL;
    if (n == 0) return BPC_OK;
    bpc_triangulate_views_kernel<<<(n + 63) / 64, 64, 0, (cudaStream_t)stream>>>(P, pts, n, V, X);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

extern "C" int bpc_detections_from_yolo(const float* xyxy, const float* conf, const float* cls, const int32_t* nraw, int SC, int Nraw,
                                        float conf_thresh, int Dmax, int32_t* boxes, double* centers, int32_t* counts, void* stream) {
    if (SC < 0 || Nraw < 1 || Dmax < 1) return BPC_EINVAL;
    if (SC > 0 && (!xyxy || !conf || !cls || !nraw || !boxes || !centers || !counts)) return BPC_EINVAL;
    if ((((uintptr_t)xyxy) & 15) != 0 || (((uintptr_t)boxes) & 15) != 0) return BPC_EALIGN;
    if (SC == 0) return BPC_OK;
    bpc_detections_kernel<<<(SC * 32 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(xyxy, conf, cls, nraw, SC, Nraw, conf_thresh, Dmax,
                                                                                    boxes, centers, counts);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

extern "C" int bpc_box_centers(const int32_t* boxes, int count, double* centers, void* stream) {
    if (count < 0 || (count > 0 && (!boxes || !centers))) return BPC_EINVAL;
    if (((uintptr_t)boxes & 15) != 0) return BPC_EALIGN;
    if (count == 0) return BPC_OK;
    bpc_box_centers_kernel<<<(count + 255) / 256, 256, 0, (cudaStream_t)stream>>>(boxes, count, centers);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

extern "C" int bpc_build_rois(const int32_t* boxes, const int32_t* idx, const int32_t* n, const int32_t* image_of_scene,
                              int S, int Dmax, int Kmax, int32_t* scene_offset, int32_t* rois, void* stream) {
    if (S < 0 || Dmax < 1 || Kmax < 1) return BPC_EINVAL;
    if (S > 0 && (!boxes || !idx || !n || !image_of_scene || !scene_offset || !rois)) return BPC_EINVAL;
    if (S == 0) return BPC_OK;
    bpc_roi_offsets_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(n, S, scene_offset);
    BPC_LAUNCH_CHECK();
    const long long total = (long long)S * Kmax * 3;
    const int blocks = (int)((total + 255) / 256 > 148 * 8 ? 148 * 8 : (total + 255) / 256);
    bpc_roi_fill_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(boxes, idx, n, image_of_scene, S, Dmax, Kmax, scene_offset, rois);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}

// ---- training-side ROI records: BOPSingleObjDataset.__getitem__, bpc/utils/data_utils.py:243-271 ----
// bbox_visib (x, y, w, h) -> the crop the dataset takes, with the scale / shift jitter of :257-271 when a draw
// is supplied (scale = 1.0 + 0.2 * random.random(), shift_x/y = random.randint(-int(0.1 w), int(0.1 w)) ...;
// the draws themselves stay on the host so that Python's `random` stream is the reference's).
namespace bpc {
__global__ void bpc_train_rois_kernel(const int32_t* __restrict__ xywh, const int32_t* __restrict__ image,
                                      const double* __restrict__ scale, const int32_t* __restrict__ shift, int n, int W, int H,
                                      int32_t* __restrict__ rois) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int x = xywh[4 * r], y = xywh[4 * r + 1], w = xywh[4 * r + 2], h = xywh[4 * r + 3];
    int x1, y1, x2, y2;
    if (scale) {
        // int(round(w * s)): Python round() of the float64 product = round-half-even (:258-259)
        int aw = (int)rint(dmul((double)w, scale[r]));
        int ah = (int)rint(dmul((double)h, scale[r]));
        const int sx = shift ? shift[2 * r] : 0, sy = shift ? shift[2 * r + 1] : 0;
        x1 = max(0, min(x - sx, W - 1));                      // :264-265
        y1 = max(0, min(y - sy, H - 1));
        aw = min(aw, W - x1);                                 // :266-267
        ah = min(ah, H - y1);
        x2 = x1 + aw; y2 = y1 + ah;
    } else {
        // bgr[y:y+h, x:x+w] (:246): NumPy clamps the slice ends to the image; starts are taken as given
        x1 = x; y1 = y; x2 = min(x + w, W); y2 = min(y + h, H);
    }
    int32_t* o = rois + 5 * (size_t)r;
    o[0] = image ? image[r] : 0; o[1] = x1; o[2] = y1; o[3] = x2; o[4] = y2;
}
}  // namespace bpc

extern "C" int bpc_train_rois(const int32_t* xywh, const int32_t* image, const double* scale, const int32_t* shift, int n,
                              int W, int H, int32_t* rois, void* stream) {
    if (n < 0 || W < 1 || H < 1) return BPC_EINVAL;
    if (n == 0) return BPC_OK;
    if (!xywh || !rois || (shift && !scale)) return BPC_EINVAL;
    bpc::bpc_train_rois_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(xywh, image, scale, shift, n, W, H, rois);
    BPC_LAUNCH_CHECK();
    return BPC_OK;
}
