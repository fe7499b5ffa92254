// Pose smoothing of a tracked video (predict.py:18-26 weighted_pts, :63-71 of the reference) as __host__ __device__
// code: project the object's 3-D box corners with a pose (utils/base_utils.py:256-265 project_points, float32 as numpy
// computes it for float32 inputs), average the recent projections, and recover a pose from the averaged corners with a
// restatement of OpenCV's cv::solvePnP(SOLVEPNP_ITERATIVE) for non-coplanar points (calib3d, cvFindExtrinsicCameraParams2:
// DLT initialisation on the normalised image points, then Levenberg-Marquardt on the pixel reprojection error).
// OpenCV stops its LM after 20 iterations or an FLT_EPSILON step; this one runs to convergence in float64, which reaches
// the same optimum (OpenCV's result sits within ~1e-9 of it on box corners).
// Only +, -, *, / and sqrt are used (no transcendental functions), and the translation unit is compiled with
// -fmad=false, so the device kernel and the *_host twin produce the same bits.
#pragma once
#include <math.h>

#include "glue_math.cuh"

namespace g6d {
namespace pnp {

constexpr int kCorners = 8;

// float32 dot product of length 3 in the order of numpy's float32 matmul (OpenBLAS sgemm: a fused multiply-add chain);
// fmaf is a single rounding on the device and in the host libm alike, so -fmad=false leaves it intact
G6D_HD float dot3_f32(float a0, float b0, float a1, float b1, float a2, float b2) {
    return fmaf(a2, b2, fmaf(a1, b1, a0 * b0));
}

// project_points for one pose: float32 [R | t] and K, pts [8,3] -> [8,2]; |depth| < 1e-4 (and != 0) becomes 1e-4
G6D_HD void project_corners(const float* pts, const float* P /* [12] */, const float* K /* [9] */, float* out /* [16] */) {
    for (int i = 0; i < kCorners; ++i) {
        const float* x = pts + i * 3;
        float c[3], p[3];
        for (int r = 0; r < 3; ++r) c[r] = dot3_f32(x[0], P[r * 4], x[1], P[r * 4 + 1], x[2], P[r * 4 + 2]) + P[r * 4 + 3];
        for (int r = 0; r < 3; ++r) p[r] = dot3_f32(c[0], K[r * 3], c[1], K[r * 3 + 1], c[2], K[r * 3 + 2]);
        float d = p[2];
        if (fabsf(d) < 1e-4f && fabsf(d) > 0.f) d = 1e-4f;
        out[i * 2] = p[0] / d;
        out[i * 2 + 1] = p[1] / d;
    }
}

// cyclic Jacobi eigen-decomposition of a symmetric n x n matrix (row-major): A's diagonal ends as the eigenvalues,
// V's columns are the eigenvectors
template <int N>
G6D_HD void jacobi_eigen(double* A, double* V) {
    for (int i = 0; i < N * N; ++i) V[i] = (i % (N + 1)) == 0 ? 1. : 0.;
    double total = 0.;
    for (int i = 0; i < N * N; ++i) total += A[i] * A[i];
    for (int sweep = 0; sweep < 64; ++sweep) {
        double off = 0.;
        for (int p = 0; p < N; ++p)
            for (int q = p + 1; q < N; ++q) off += A[p * N + q] * A[p * N + q];
        if (off <= 1e-34 * total) break;
        for (int p = 0; p < N; ++p)
            for (int q = p + 1; q < N; ++q) {
                const double apq = A[p * N + q];
                if (apq == 0.) continue;
                const double theta = (A[q * N + q] - A[p * N + p]) / (2. * apq);
                double t = 1. / (fabs(theta) + sqrt(theta * theta + 1.));
                if (fabs(theta) > 1e150) t = 0.5 / fabs(theta);
                if (theta < 0.) t = -t;
                const double c = 1. / sqrt(t * t + 1.), s = t * c;
                for (int k = 0; k < N; ++k) {                         // A <- A G (columns p, q)
                    const double akp = A[k * N + p], akq = A[k * N + q];
                    A[k * N + p] = c * akp - s * akq;
                    A[k * N + q] = s * akp + c * akq;
                }
                for (int k = 0; k < N; ++k) {                         // A <- G^T A (rows p, q)
                    const double apk = A[p * N + k], aqk = A[q * N + k];
                    A[p * N + k] = c * apk - s * aqk;
                    A[q * N + k] = s * apk + c * aqk;
                }
                for (int k = 0; k < N; ++k) {
                    const double vkp = V[k * N + p], vkq = V[k * N + q];
                    V[k * N + p] = c * vkp - s * vkq;
                    V[k * N + q] = s * vkp + c * vkq;
                }
            }
    }
}

G6D_HD double det3(const double* m) {
    return m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
}

// orthogonal polar factor U V^T of a non-singular 3x3 (cv::SVD's U V^T in the DLT initialisation): Newton's iteration
// X <- (X + X^-T) / 2 from X scaled to unit Frobenius norm per row
G6D_HD void polar3(const double* M, double* R) {
    double n = 0.;
    for (int i = 0; i < 9; ++i) n += M[i] * M[i];
    const double s = sqrt(3. / n);
    for (int i = 0; i < 9; ++i) R[i] = M[i] * s;
    for (int it = 0; it < 100; ++it) {
        double Ri[9], d = 0.;
        glue::inv3_cv(R, Ri);
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                const double v = 0.5 * (R[i * 3 + j] + Ri[j * 3 + i]);
                d = fmax(d, fabs(v - R[i * 3 + j]));
                R[i * 3 + j] = v;
            }
        if (d < 1e-15) break;
    }
}

// pixel residuals (projection - m) [16] and, optionally, their Jacobian [16,6] w.r.t. a left rotation increment w
// (R <- exp([w]x) R) and t
G6D_HD double residuals(const double* X, const double* m, const double* K, const double* R, const double* t, double* res, double* J) {
    double cost = 0.;
    for (int i = 0; i < kCorners; ++i) {
        double w[3], c[3], p[3];
        glue::mat3_vec(R, X + i * 3, w);
        for (int r = 0; r < 3; ++r) c[r] = w[r] + t[r];
        glue::mat3_vec(K, c, p);
        const double u = p[0] / p[2], v = p[1] / p[2];
        res[i * 2] = u - m[i * 2];
        res[i * 2 + 1] = v - m[i * 2 + 1];
        cost += res[i * 2] * res[i * 2] + res[i * 2 + 1] * res[i * 2 + 1];
        if (!J) continue;
        for (int k = 0; k < 2; ++k) {
            const double uv = k == 0 ? u : v;
            double a[3];                                              // d(u or v) / d(camera point)
            for (int e = 0; e < 3; ++e) a[e] = (K[k * 3 + e] - uv * K[6 + e]) / p[2];
            double* row = J + (i * 2 + k) * 6;
            row[0] = w[1] * a[2] - w[2] * a[1];                       // d/dw = w x a  (d camera point / dw = -[w]x)
            row[1] = w[2] * a[0] - w[0] * a[2];
            row[2] = w[0] * a[1] - w[1] * a[0];
            row[3] = a[0]; row[4] = a[1]; row[5] = a[2];
        }
    }
    return cost;
}

// solve the 6x6 symmetric positive definite system A x = b (Cholesky); false when A is not positive definite
G6D_HD bool solve6(const double* A, const double* b, double* x) {
    double L[36] = {0.};
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j <= i; ++j) {
            double s = A[i * 6 + j];
            for (int k = 0; k < j; ++k) s -= L[i * 6 + k] * L[j * 6 + k];
            if (i == j) {
                if (!(s > 0.)) return false;
                L[i * 6 + i] = sqrt(s);
            } else {
                L[i * 6 + j] = s / L[j * 6 + j];
            }
        }
    double y[6];
    for (int i = 0; i < 6; ++i) {
        double s = b[i];
        for (int k = 0; k < i; ++k) s -= L[i * 6 + k] * y[k];
        y[i] = s / L[i * 6 + i];
    }
    for (int i = 5; i >= 0; --i) {
        double s = y[i];
        for (int k = i + 1; k < 6; ++k) s -= L[k * 6 + i] * x[k];
        x[i] = s / L[i * 6 + i];
    }
    return true;
}

// R <- rotation of the quaternion (1, w / 2) (normalised) @ R
G6D_HD void rotate_left(const double* w, const double* R, double* out) {
    double qw = 1., qx = 0.5 * w[0], qy = 0.5 * w[1], qz = 0.5 * w[2];
    const double n = sqrt(qw * qw + qx * qx + qy * qy + qz * qz);
    qw /= n; qx /= n; qy /= n; qz /= n;
    const double Q[9] = {1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qw * qz), 2 * (qx * qz + qw * qy),
                         2 * (qx * qy + qw * qz), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qw * qx),
                         2 * (qx * qz - qw * qy), 2 * (qy * qz + qw * qx), 1 - 2 * (qx * qx + qy * qy)};
    glue::mat3_mul(Q, R, out);
}

// SOLVEPNP_ITERATIVE for 8 non-coplanar points: X [8,3] object points, m [8,2] pixels, K [9] -> pose [12] = [R | t]
G6D_HD void solve_pnp(const double* X, const double* m, const double* K, double* pose) {
    // normalised image points (cv::undistortPoints with zero distortion)
    double Ki[9], mn[kCorners * 2];
    glue::inv3_cv(K, Ki);
    for (int i = 0; i < kCorners; ++i) {
        const double v[3] = {m[i * 2], m[i * 2 + 1], 1.};
        double q[3];
        glue::mat3_vec(Ki, v, q);
        mn[i * 2] = q[0] / q[2];
        mn[i * 2 + 1] = q[1] / q[2];
    }
    // DLT: the [3,4] matrix minimising |L p| is the eigenvector of L^T L with the smallest eigenvalue
    double LL[144] = {0.}, V[144];
    for (int i = 0; i < kCorners; ++i) {
        const double* M = X + i * 3;
        double rows[2][12];
        for (int k = 0; k < 2; ++k) {
            const double s = -mn[i * 2 + k];
            for (int e = 0; e < 12; ++e) rows[k][e] = 0.;
            for (int e = 0; e < 3; ++e) { rows[k][k * 4 + e] = M[e]; rows[k][8 + e] = s * M[e]; }
            rows[k][k * 4 + 3] = 1.;
            rows[k][11] = s;
        }
        for (int k = 0; k < 2; ++k)
            for (int a = 0; a < 12; ++a)
                for (int b = 0; b < 12; ++b) LL[a * 12 + b] += rows[k][a] * rows[k][b];
    }
    jacobi_eigen<12>(LL, V);
    int best = 0;
    for (int e = 1; e < 12; ++e)
        if (LL[e * 13] < LL[best * 13]) best = e;
    double RRt[12];
    for (int e = 0; e < 12; ++e) RRt[e] = V[e * 12 + best];
    double RR[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) RR[i * 3 + j] = RRt[i * 4 + j];
    if (det3(RR) < 0.) {
        for (int e = 0; e < 12; ++e) RRt[e] = -RRt[e];
        for (int e = 0; e < 9; ++e) RR[e] = -RR[e];
    }
    double sc = 0.;
    for (int e = 0; e < 9; ++e) sc += RR[e] * RR[e];
    sc = sqrt(sc);
    double R[9], t[3];
    polar3(RR, R);
    double nr = 0.;
    for (int e = 0; e < 9; ++e) nr += R[e] * R[e];
    for (int i = 0; i < 3; ++i) t[i] = RRt[i * 4 + 3] * (sqrt(nr) / sc);
    // Levenberg-Marquardt on the pixel reprojection error
    double res[kCorners * 2], J[kCorners * 2 * 6];
    double cost = residuals(X, m, K, R, t, res, J);
    double lambda = 1e-3;
    for (int it = 0; it < 200 && lambda < 1e12; ++it) {
        double A[36], g[6];
        for (int a = 0; a < 6; ++a) {
            g[a] = 0.;
            for (int r = 0; r < kCorners * 2; ++r) g[a] -= J[r * 6 + a] * res[r];
            for (int b = 0; b < 6; ++b) {
                double s = 0.;
                for (int r = 0; r < kCorners * 2; ++r) s += J[r * 6 + a] * J[r * 6 + b];
                A[a * 6 + b] = s;
            }
        }
        for (int a = 0; a < 6; ++a) A[a * 7] += lambda * A[a * 7];
        double d[6];
        if (!solve6(A, g, d)) { lambda *= 10.; continue; }
        double Rn[9], tn[3], rn[kCorners * 2];
        rotate_left(d, R, Rn);
        for (int i = 0; i < 3; ++i) tn[i] = t[i] + d[3 + i];
        const double cn = residuals(X, m, K, Rn, tn, rn, nullptr);
        if (cn < cost) {
            double step = 0., size = 1.;
            for (int a = 0; a < 6; ++a) step += d[a] * d[a];
            for (int i = 0; i < 3; ++i) size += t[i] * t[i];
            for (int e = 0; e < 9; ++e) R[e] = Rn[e];
            for (int i = 0; i < 3; ++i) t[i] = tn[i];
            cost = residuals(X, m, K, R, t, res, J);
            lambda = fmax(lambda * 0.1, 1e-12);
            if (step < 1e-30 * size) break;
        } else {
            lambda *= 10.;
        }
    }
    for (int i = 0; i < 3; ++i) {
        pose[i * 4] = R[i * 3]; pose[i * 4 + 1] = R[i * 3 + 1]; pose[i * 4 + 2] = R[i * 3 + 2];
        pose[i * 4 + 3] = t[i];
    }
}

// one lane of g6d_track_smooth
G6D_HD void track_smooth_lane(int l, const float* bbox, const double* poses, const g6d_glue_camera* cams, const double* weights,
                              const double* wsum, int num, float* hist, int* count, float* corners, double* wpts, double* smoothed) {
    float P[12], Kf[9];
    for (int e = 0; e < 12; ++e) P[e] = (float)poses[(long long)l * 12 + e];
    for (int e = 0; e < 9; ++e) Kf[e] = (float)cams[l].K[e];
    float c[kCorners * 2];
    project_corners(bbox, P, Kf, c);
    const int cnt = count[l];
    float* h = hist + (long long)l * num * kCorners * 2;
    for (int e = 0; e < kCorners * 2; ++e) {
        h[(cnt % num) * kCorners * 2 + e] = c[e];
        corners[(long long)l * kCorners * 2 + e] = c[e];
    }
    const int total = cnt + 1, n = total < num ? total : num;
    count[l] = total;
    // np.sum(np.asarray(pts_list) * weights[:, None, None], 0) / np.sum(weights): oldest first, float64
    double w[kCorners * 2];
    for (int j = 0; j < n; ++j) {
        const float* s = h + ((total - n + j) % num) * kCorners * 2;
        const double wj = weights[num - n + j];
        for (int e = 0; e < kCorners * 2; ++e) w[e] = j == 0 ? (double)s[e] * wj : w[e] + (double)s[e] * wj;
    }
    for (int e = 0; e < kCorners * 2; ++e) {
        w[e] = w[e] / wsum[n - 1];
        wpts[(long long)l * kCorners * 2 + e] = w[e];
    }
    double X[kCorners * 3];
    for (int e = 0; e < kCorners * 3; ++e) X[e] = (double)bbox[e];
    solve_pnp(X, w, cams[l].K, smoothed + (long long)l * 12);
}

}  // namespace pnp
}  // namespace g6d
