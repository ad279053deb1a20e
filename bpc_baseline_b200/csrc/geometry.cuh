// Per-scene epipolar geometry in shared memory: fundamental matrices, projection matrices,
// normalised epipolar lines per detection, pair distances and the (virtual) cost tensor.
//
// Reference: bpc/inference/utils/camera_utils.py:23-46 (F), bpc/inference/epipolar_matching.py:5-28
// (symmetric epipolar distance), :73-81 (three-pair mean), bpc/inference/process_pose.py:88-92 (P).
#pragma once
#include "common.cuh"

namespace bpc {

// ---- float32 inverse of K (np.linalg.inv on a float32 3x3, camera_utils.py:38-39) -------------------
// numpy.linalg.inv computes in DOUBLE whatever the input type (numpy/linalg/_linalg.py: _commonType returns
// `double` as the computation type, the 'd->d' gufunc = LAPACK dgesv runs, and the result is cast back with
// astype(float32)), so the float32 inverse is the correctly rounded exact inverse up to double rounding.
// Checked against np.linalg.inv: 3000 / 3000 skewed K bit-equal to float32(exact); golden tests/golden/skew.npz.
__device__ inline void inv3_f32(const float* K, float* Ki) {
    if (K[1] == 0.f && K[3] == 0.f && K[6] == 0.f && K[7] == 0.f && K[8] == 1.f) {
        // zero-skew pinhole: the exact entries are single quotients, and a float32 division is their correct rounding
        // (bit-identical to np.linalg.inv on 20 000 / 20 000 random pinhole K, SURVEY.md a1)
        const float fx = K[0], fy = K[4], cx = K[2], cy = K[5];
        Ki[0] = __fdiv_rn(1.f, fx); Ki[1] = 0.f; Ki[2] = __fdiv_rn(-cx, fx);
        Ki[3] = 0.f; Ki[4] = __fdiv_rn(1.f, fy); Ki[5] = __fdiv_rn(-cy, fy);
        Ki[6] = 0.f; Ki[7] = 0.f; Ki[8] = 1.f;
        return;
    }
    // general K: float64 Gauss-Jordan with partial pivoting (dgesv's pivot choice), rounded to float32 at the end
    double a[3][6];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) { a[r][c] = (double)K[r * 3 + c]; a[r][3 + c] = (r == c) ? 1.0 : 0.0; }
    for (int col = 0; col < 3; ++col) {
        int piv = col;
        for (int r = col + 1; r < 3; ++r)
            if (fabs(a[r][col]) > fabs(a[piv][col])) piv = r;
        if (piv != col)
            for (int c = 0; c < 6; ++c) { const double t = a[col][c]; a[col][c] = a[piv][c]; a[piv][c] = t; }
        const double d = a[col][col];
        for (int c = 0; c < 6; ++c) a[col][c] = ddiv(a[col][c], d);
        for (int r = 0; r < 3; ++r) {
            if (r == col) continue;
            const double f = a[r][col];
            for (int c = 0; c < 6; ++c) a[r][c] = dfma(-f, a[col][c], a[r][c]);
        }
    }
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) Ki[r * 3 + c] = __double2float_rn(a[r][3 + c]);
}

// ---- compute_fundamental_matrix(K1, R1, t1, K2, R2, t2), camera_utils.py:23-46 ----------------------
// K: float32 3x3; RT: float64 4x4 (R = RT[:3,:3], t = RT[:3,3], process_pose.py:155-156).
__device__ inline void fundamental(const float* K1, const double* RT1, const float* K2, const double* RT2, double* F) {
    double Rr[9];
    for (int r = 0; r < 3; ++r)          // R_rel = R2 @ R1.T   (:27)
        for (int c = 0; c < 3; ++c)
            Rr[r * 3 + c] = dot3_seq(RT2[r * 4 + 0], RT1[c * 4 + 0], RT2[r * 4 + 1], RT1[c * 4 + 1],
                                     RT2[r * 4 + 2], RT1[c * 4 + 2]);
    double tr[3];
    for (int r = 0; r < 3; ++r)          // t_rel = t2 - R_rel @ t1   (:28)
        tr[r] = dsub(RT2[r * 4 + 3], dot3_gemv(Rr[r * 3 + 0], RT1[3], Rr[r * 3 + 1], RT1[7], Rr[r * 3 + 2], RT1[11]));
    // [t]x rounded to float32 (:31-35)
    const double t0 = (double)__double2float_rn(tr[0]);
    const double t1 = (double)__double2float_rn(tr[1]);
    const double t2 = (double)__double2float_rn(tr[2]);
    const double tx[9] = {0.0, -t2, t1, t2, 0.0, -t0, -t1, t0, 0.0};
    double E[9];
    for (int r = 0; r < 3; ++r)          // E = tx @ R_rel   (:37)
        for (int c = 0; c < 3; ++c)
            E[r * 3 + c] = dot3_seq(tx[r * 3 + 0], Rr[0 + c], tx[r * 3 + 1], Rr[3 + c], tx[r * 3 + 2], Rr[6 + c]);
    float K1i[9], K2i[9];
    inv3_f32(K1, K1i);
    inv3_f32(K2, K2i);
    double Mx[9];
    for (int r = 0; r < 3; ++r)          // K2_inv.T @ E   (:40, left to right)
        for (int c = 0; c < 3; ++c)
            Mx[r * 3 + c] = dot3_seq((double)K2i[0 + r], E[0 + c], (double)K2i[3 + r], E[3 + c], (double)K2i[6 + r], E[6 + c]);
    for (int r = 0; r < 3; ++r)          // (...) @ K1_inv
        for (int c = 0; c < 3; ++c)
            F[r * 3 + c] = dot3_seq(Mx[r * 3 + 0], (double)K1i[0 + c], Mx[r * 3 + 1], (double)K1i[3 + c],
                                    Mx[r * 3 + 2], (double)K1i[6 + c]);
    const double f22 = F[8];
    if (fabs(f22) > 1e-8)                // (:43-44)
        for (int e = 0; e < 9; ++e) F[e] = ddiv(F[e], f22);
}

// P = K (float32) @ RT[:3] (float64), process_pose.py:91
__device__ inline void projection(const float* K, const double* RT, double* Pm) {
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 4; ++c)
            Pm[r * 4 + c] = dot3_seq((double)K[r * 3 + 0], RT[0 + c], (double)K[r * 3 + 1], RT[4 + c],
                                     (double)K[r * 3 + 2], RT[8 + c]);
}

// Normalised epipolar line of one point (epipolar_matching.py:13-23).
//   transpose == 0: l = F   @ (x, y, 1)  -- "l2", the line in the second camera of the pair
//   transpose == 1: l = F.T @ (x, y, 1)  -- "l1", the line in the first camera
// Returns false when the norm of (a, b) is <= 1e-8 (the caller then uses the 9999 sentinel).
__device__ inline bool epiline(const double* F, int transpose, double x, double y, double* l) {
    if (!transpose) {
        for (int r = 0; r < 3; ++r) l[r] = dot3_gemv(F[r * 3 + 0], x, F[r * 3 + 1], y, F[r * 3 + 2], 1.0);
    } else {
        for (int c = 0; c < 3; ++c) l[c] = dot3_seq(F[0 + c], x, F[3 + c], y, F[6 + c], 1.0);
    }
    const double nrm = sqrt(dfma(l[1], l[1], dmul(l[0], l[0])));   // np.linalg.norm(l[:2])
    if (nrm > 1e-8) {
        l[0] = ddiv(l[0], nrm); l[1] = ddiv(l[1], nrm); l[2] = ddiv(l[2], nrm);
        return true;
    }
    return false;
}

__device__ __forceinline__ double line_point(const double* l, double x, double y) {
    return fabs(dot3_seq(l[0], x, l[1], y, l[2], 1.0));            // abs(np.dot(l, pt_h))
}

// Scene state resident in shared memory.
struct Scene {
    double* pts;       // [3][Dmax][2]
    double* lines;     // [6][Dmax][3]   0:l2_12[i] 1:l1_12[j] 2:l2_13[i] 3:l1_13[k] 4:l2_23[j] 5:l1_23[k]
    uint8_t* lvalid;   // [6][Dmax]
    int N, M, P, Dmax;
    unsigned long long m_magic;   // 2^40 / M + 1: r / M == (r * m_magic) >> 40 for r * M < 2^40

    __device__ __forceinline__ const double* pt(int cam, int d) const { return pts + ((size_t)cam * Dmax + d) * 2; }
    __device__ __forceinline__ const double* line(int set, int d) const { return lines + ((size_t)set * Dmax + d) * 3; }
    __device__ __forceinline__ bool valid(int set, int d) const { return lvalid[set * Dmax + d] != 0; }

    // epipolar_error(pa, pb, F_ab): 0.5 * (d1 + d2), d = 9999 when its line is degenerate (:25-28)
    __device__ __forceinline__ double pair(int set_l2, int set_l1, int cam_a, int a, int cam_b, int b) const {
        const double* pa = pt(cam_a, a);
        const double* pb = pt(cam_b, b);
        // a degenerate line is stored as (0, 0, 9999): |fma(9999, 1, fma(0, y, 0 * x))| = 9999 exactly for finite x, y,
        // i.e. the sentinel of :25-26 without a validity load and select per evaluation
        const double d1 = line_point(line(set_l1, b), pa[0], pa[1]);
        const double d2 = line_point(line(set_l2, a), pb[0], pb[1]);
        return dmul(0.5, dadd(d1, d2));
    }
    __device__ __forceinline__ double e12(int i, int j) const { return pair(0, 1, 0, i, 1, j); }
    __device__ __forceinline__ double e13(int i, int k) const { return pair(2, 3, 0, i, 2, k); }
    __device__ __forceinline__ double e23(int j, int k) const { return pair(4, 5, 1, j, 2, k); }
    // (e12 + e13 + e23) before the division by 3 (:81)
    __device__ __forceinline__ double sum3(int i, int j, int k) const { return dadd(dadd(e12(i, j), e13(i, k)), e23(j, k)); }
    __device__ __forceinline__ float cost(int i, int j, int k) const { return cost_from_sum(sum3(i, j, k)); }
};

// Fill pts / lines / lvalid of a scene from global memory.  All threads of the CTA call it; the
// caller must __syncthreads() afterwards.  F = [3][9] (12, 13, 23), already in shared memory.
// Returns true when this thread loaded a point with a coordinate that is not below 1e300 in magnitude, or a line with a
// component that is not finite.  Without any such input no pair distance can be NaN: every line component is finite and
// |a|, |b| <= 1 (or the sentinel / zero line), so no product in |a x + b y + c| overflows and no inf - inf can occur.
__device__ inline bool scene_load(Scene& sc, const double* F, const double* centers_scene, int nthreads, int tid) {
    const int D = sc.Dmax;
    const int cnt[3] = {sc.N, sc.M, sc.P};
    bool suspect = false;
    for (int e = tid; e < 3 * D; e += nthreads) {
        const int cam = e / D, d = e - cam * D;
        if (d < cnt[cam]) {
            const double x = centers_scene[(size_t)e * 2 + 0], y = centers_scene[(size_t)e * 2 + 1];
            sc.pts[(size_t)e * 2 + 0] = x;
            sc.pts[(size_t)e * 2 + 1] = y;
            suspect |= !(fabs(x) < 1e300) || !(fabs(y) < 1e300);
        }
    }
    // set -> (F index, transpose, camera of the point)
    const int set_F[6] = {0, 0, 1, 1, 2, 2};
    const int set_T[6] = {0, 1, 0, 1, 0, 1};
    const int set_cam[6] = {0, 1, 0, 2, 1, 2};
    for (int e = tid; e < 6 * D; e += nthreads) {
        const int set = e / D, d = e - set * D;
        const int cam = set_cam[set];
        if (d >= cnt[cam]) continue;
        const double* p = centers_scene + ((size_t)cam * D + d) * 2;
        double l[3];
        const bool ok = epiline(F + set_F[set] * 9, set_T[set], p[0], p[1], l);
        double* dst = sc.lines + (size_t)e * 3;
        dst[0] = ok ? l[0] : 0.0; dst[1] = ok ? l[1] : 0.0; dst[2] = ok ? l[2] : 9999.0;
        sc.lvalid[e] = ok ? 1 : 0;
        const double INF = __longlong_as_double(0x7ff0000000000000LL);
        suspect |= !(fabs(dst[0]) < INF) || !(fabs(dst[1]) < INF) || !(fabs(dst[2]) < INF);
    }
    return suspect;
}

// ---- DLT triangulation of one 3-view match (epipolar_matching.py:118-127) ---------------------------
// Rows x*P[2]-P[0], y*P[2]-P[1] per view -> A (6x4); X = right singular vector of the smallest singular
// value, dehomogenised.  One-sided (Hestenes) Jacobi in float64, register resident.
__device__ inline void triangulate3(const double* Pm /*[3][12]*/, const double* xy /*[3][2]*/, double* X) {
    double A[6][4], V[4][4];
#pragma unroll
    for (int v = 0; v < 3; ++v) {
        const double x = xy[v * 2 + 0], y = xy[v * 2 + 1];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            A[2 * v][c] = dsub(dmul(x, Pm[v * 12 + 8 + c]), Pm[v * 12 + 0 + c]);
            A[2 * v + 1][c] = dsub(dmul(y, Pm[v * 12 + 8 + c]), Pm[v * 12 + 4 + c]);
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) V[r][c] = (r == c) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 16; ++sweep) {
        bool rotated = false;
#pragma unroll
        for (int p = 0; p < 3; ++p) {
#pragma unroll
            for (int q = p + 1; q < 4; ++q) {
                double alpha = 0.0, beta = 0.0, gamma = 0.0;
#pragma unroll
                for (int r = 0; r < 6; ++r) {
                    alpha += A[r][p] * A[r][p];
                    beta += A[r][q] * A[r][q];
                    gamma += A[r][p] * A[r][q];
                }
                if (fabs(gamma) > 1e-15 * sqrt(alpha * beta) && fabs(gamma) > 1e-300) {
                    const double zeta = (beta - alpha) / (2.0 * gamma);
                    double t;
                    if (fabs(zeta) > 1e150) t = 0.5 / zeta;
                    else t = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                    const double c = 1.0 / sqrt(1.0 + t * t);
                    const double s = c * t;
#pragma unroll
                    for (int r = 0; r < 6; ++r) {
                        const double ap = A[r][p], aq = A[r][q];
                        A[r][p] = c * ap - s * aq;
                        A[r][q] = s * ap + c * aq;
                    }
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const double vp = V[r][p], vq = V[r][q];
                        V[r][p] = c * vp - s * vq;
                        V[r][q] = s * vp + c * vq;
                    }
                    rotated = true;
                }
            }
        }
        if (!rotated) break;
    }
    double best = 0.0;
    int bi = 0;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        double nrm = 0.0;
#pragma unroll
        for (int r = 0; r < 6; ++r) nrm += A[r][c] * A[r][c];
        if (c == 0 || nrm < best) { best = nrm; bi = c; }
    }
    double h[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        double v = V[r][0];
        if (bi == 1) v = V[r][1];
        if (bi == 2) v = V[r][2];
        if (bi == 3) v = V[r][3];
        h[r] = v;
    }
    X[0] = h[0] / h[3];
    X[1] = h[1] / h[3];
    X[2] = h[2] / h[3];
}

// compute_reprojection_error(P, X, pt), utils/triangulation.py:14-18
__device__ inline double reprojection(const double* Pm /*[12]*/, const double* X, const double* xy) {
    double pr[3];
    for (int r = 0; r < 3; ++r)
        pr[r] = Pm[r * 4 + 0] * X[0] + Pm[r * 4 + 1] * X[1] + Pm[r * 4 + 2] * X[2] + Pm[r * 4 + 3];
    const double u = pr[0] / pr[2] - xy[0];
    const double v = pr[1] / pr[2] - xy[1];
    return sqrt(u * u + v * v);
}

}  // namespace bpc
