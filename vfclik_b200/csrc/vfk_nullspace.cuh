// vfk_nullspace.cuh -- rare-path dense linear algebra: orthonormal basis of null(J) for the reference's nullspace control
// interface (Householder QR), and a one-sided Jacobi SVD shared by the undamped projector and the truncated velocity IK.
//
// scripts/nullspace:75-107 builds B = I - pinv(J) J (LAPACK SVD) and takes the left singular vectors of B^T whose
// singular value is >= 1e-8: an orthonormal basis of null(J), k = N - rank(J) vectors.  Forming B through the normal
// equations J^T (J J^T)^-1 J loses cond(J)^2 * eps; a Householder QR of J^T (N x 6) loses only cond(J) * eps and needs
// no damping: J^T = Q R, Q = H_0 ... H_5 orthogonal N x N, and columns 6 .. N-1 of Q are orthogonal to range(J^T),
// i.e. they span null(J) (exactly N - 6 of them when J has full row rank; at a rank-deficient posture they are still
// null vectors, the reference would find one more).  The reflectors follow LAPACK's dgeqr2 / dlarfg convention
// (beta = -sign(alpha) |x|, v_0 = 1, H = I - tau v v^T), so numpy.linalg.qr(J.T, mode="complete") gives the same
// vectors up to rounding -- that is what oracle/batch.py:ns_basis pins this against.
//
// The projector (I - pinv(J) J) x does not use that basis: Q diag(0, .., 0, 1, .., 1) Q^T x projects onto N - 6
// dimensions, and at a posture where J loses rank (rank r < 6) null(J) has N - r.  It goes through the singular values
// instead (ns_svd_project): rank-revealing, with the cutoff of numpy's pinv that the reference calls.
//
// Rare path (control mode / undamped projector / truncated IK), any N <= 17: rolled loops over thread-local arrays,
// compiled once per translation unit and called -- it costs the throughput instantiations neither registers nor
// instruction-cache lines.
#pragma once
#include <cuda_runtime.h>
#include <math.h>

namespace vfk {

// Factor a = J^T, n x 6 row-major (a[r * 6 + c] = J[c][r]), in place: on return the reflector vectors sit below the
// diagonal (v_j[j] = 1 implied) and tau[j] holds their scales; tau[j] = 0 means H_j = I (dlarfg's zero-tail case, and every
// j >= n).
static __device__ __noinline__ void ns_qr_factor(double* a, int n, double* tau) {
    for (int j = 0; j < 6; ++j) {
        tau[j] = 0.0;
        if (j >= n) continue;
        const double alpha = a[j * 6 + j];
        double xn2 = 0.0;
        for (int r = j + 1; r < n; ++r) xn2 = fma(a[r * 6 + j], a[r * 6 + j], xn2);
        if (xn2 == 0.0) continue;
        const double beta = -copysign(sqrt(fma(alpha, alpha, xn2)), alpha);
        tau[j] = (beta - alpha) / beta;
        const double sc = 1.0 / (alpha - beta);
        for (int r = j + 1; r < n; ++r) a[r * 6 + j] *= sc;
        a[j * 6 + j] = beta;
        for (int c = j + 1; c < 6; ++c) {                          // apply H_j to the remaining columns
            double w = a[j * 6 + c];
            for (int r = j + 1; r < n; ++r) w = fma(a[r * 6 + j], a[r * 6 + c], w);
            w *= tau[j];
            a[j * 6 + c] -= w;
            for (int r = j + 1; r < n; ++r) a[r * 6 + c] = fma(-a[r * 6 + j], w, a[r * 6 + c]);
        }
    }
}

__device__ __forceinline__ void ns_reflect(const double* a, double tau_j, int j, int n, double* w) {
    if (tau_j == 0.0) return;
    double d = w[j];
    for (int r = j + 1; r < n; ++r) d = fma(a[r * 6 + j], w[r], d);
    d *= tau_j;
    w[j] -= d;
    for (int r = j + 1; r < n; ++r) w[r] = fma(-a[r * 6 + j], d, w[r]);
}

// w <- Q e_col = H_0 ( ... (H_5 e_col)): column `col` of Q; col >= 6 is a unit vector of null(J).
static __device__ __noinline__ void ns_qr_column(const double* a, const double* tau, int n, int col, double* w) {
    for (int r = 0; r < n; ++r) w[r] = (r == col) ? 1.0 : 0.0;
    for (int j = 5; j >= 0; --j) ns_reflect(a, tau[j], j, n, w);
}

// ---- one-sided Jacobi SVD (Hestenes), same rare-path style.
// g: 6 x n row-major (g[r * n + j]).  Plane rotations of row pairs until the rows are mutually orthogonal: on return
// g = U^T G = Sigma V^T, row i being sigma_i v_i^T, which resolves every singular value to relative accuracy (no squaring
// of the condition number).  y (6 values, or null) receives the same rotations: U^T y.
static __device__ __noinline__ void jacobi_rows(double* g, int n, double* y) {
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0;
        for (int p = 0; p < 5; ++p)
            for (int q = p + 1; q < 6; ++q) {
                double a = 0.0, b = 0.0, c = 0.0;
                for (int j = 0; j < n; ++j) {
                    a = fma(g[p * n + j], g[p * n + j], a);
                    b = fma(g[q * n + j], g[q * n + j], b);
                    c = fma(g[p * n + j], g[q * n + j], c);
                }
                const double scale = sqrt(a * b);
                if (!(fabs(c) > 1e-17 * scale) || scale == 0.0) continue;
                off = fmax(off, fabs(c) / scale);
                const double zeta = (b - a) / (2.0 * c);
                const double t = copysign(1.0, zeta) / (fabs(zeta) + sqrt(fma(zeta, zeta, 1.0)));
                const double cs = 1.0 / sqrt(fma(t, t, 1.0)), sn = cs * t;
                for (int j = 0; j < n; ++j) {
                    const double u = g[p * n + j], v = g[q * n + j];
                    g[p * n + j] = cs * u - sn * v;
                    g[q * n + j] = sn * u + cs * v;
                }
                if (y) {
                    const double u = y[p], v = y[q];
                    y[p] = cs * u - sn * v;
                    y[q] = sn * u + cs * v;
                }
            }
        if (off < 1e-15) break;
    }
}

// Relative cutoff of the undamped projector: singular values sigma_i <= cut * sigma_max count as zero.  FP64: 1e-15, the
// default of numpy.linalg.pinv and so the reference's own rule (scripts/nullspace:78).  FP32: the Jacobian is rounded to
// float (6e-8 relative) before this FP64 factorisation, which lifts an exactly zero singular value to ~1e-9 .. 1e-8 of
// sigma_max; with 1e-15 those would count as rank and turn the projector O(1) wrong.  Any cutoff in 1e-7 .. 1e-5 cuts
// them: at exactly singular LWR postures the projector of the rounded Jacobian then matches the FP64 one to 2e-7.  Near
// a singularity (cond(J) ~ 1e6) the FP32 projector is O(1) off either way (DESIGN.md section 2).
constexpr double kNsCutF64 = 1e-15, kNsCutF32 = 1e-6;

// w <- (I - pinv(J) J) w, g = J (6 x n row-major, destroyed): after jacobi_rows row i of g is sigma_i v_i^T, so
// pinv(J) J = sum over sigma_i > cut * sigma_max of v_i v_i^T, and w loses its component g_i (g_i . w) / |g_i|^2 along
// each kept row.  Rank-revealing: at rank r < 6 the result lies in the whole (N - r)-dimensional null(J).
static __device__ __noinline__ void ns_svd_project(double* g, int n, double cut, double* w) {
    jacobi_rows(g, n, nullptr);
    double s2[6], smax2 = 0.0;
    for (int r = 0; r < 6; ++r) {
        s2[r] = 0.0;
        for (int j = 0; j < n; ++j) s2[r] = fma(g[r * n + j], g[r * n + j], s2[r]);
        smax2 = fmax(smax2, s2[r]);
    }
    const double cut2 = cut * cut * smax2;
    for (int r = 0; r < 6; ++r) {
        if (!(s2[r] > cut2)) continue;
        double d = 0.0;
        for (int j = 0; j < n; ++j) d = fma(g[r * n + j], w[j], d);
        d /= s2[r];
        for (int j = 0; j < n; ++j) w[j] = fma(-d, g[r * n + j], w[j]);
    }
}

// ---- truncated weighted least squares (VFK_IK_TRUNCATED).
// g: Jw = Wt J Wj, 6 x n row-major (g[r * n + j]); y: Wt t (6).  jacobi_rows gives G' = U^T Jw = Sigma V^T and U^T y, so
//   qd = V diag(f(sigma)) U^T y = sum_i row_i * c_i * (U^T y)_i,  c_i = 1 / sigma_i^2 (sigma_i >= eps), 1 / (sigma_i^2 + lambda^2) below.
// qd: n values (before the joint weights).  Restated by oracle/batch.py:ikv_dls (ik_mode 1) through numpy's SVD.
static __device__ __noinline__ void ik_truncated(double* g, int n, double* y, double lambda2, double eps, double* qd) {
    jacobi_rows(g, n, y);
    for (int j = 0; j < n; ++j) qd[j] = 0.0;
    const double eps2 = eps * eps;
    for (int r = 0; r < 6; ++r) {
        double s2 = 0.0;
        for (int j = 0; j < n; ++j) s2 = fma(g[r * n + j], g[r * n + j], s2);
        if (s2 == 0.0) continue;
        const double coef = y[r] / (s2 >= eps2 ? s2 : s2 + lambda2);
        for (int j = 0; j < n; ++j) qd[j] = fma(coef, g[r * n + j], qd[j]);
    }
}

// vectors of the basis the four-float control interface can address: min(4, N - 6) (scripts/nullspace:113)
__host__ __device__ constexpr int ns_ctrl_vectors(int n) { return n > 6 ? (n - 6 < 4 ? n - 6 : 4) : 0; }
__host__ __device__ constexpr int ns_null_vectors(int n) { return n > 6 ? n - 6 : 0; }

}  // namespace vfk
