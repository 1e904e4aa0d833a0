// 3x3 double helpers shared by the device pipeline (K5/K6) and the host-side static API
// (vstab_decompose_homography / vstab_compose_homography).
//   decompose_h  <- Stabilizer::decomposeHomography  /root/reference/src/stabilizer.cpp:1435-1533
//                   (+ qrDecomposition2x2 :1342-1432, whose throws become `false`, SURVEY B.14)
//   compose_h    <- Stabilizer::composeHomography    /root/reference/src/stabilizer.cpp:1535-1566
//   invert3      <- cv::invert(3x3, DECOMP_LU) closed form (cofactors / determinant)
#pragma once
#include <math.h>
#include "common.cuh"

namespace vstabk {

struct HParams {
    double s, theta, k, delta, t[2], v[2];
};

VSTAB_HD void eye3(double* H) {
    H[0] = 1; H[1] = 0; H[2] = 0; H[3] = 0; H[4] = 1; H[5] = 0; H[6] = 0; H[7] = 0; H[8] = 1;
}

VSTAB_HD void matmul3(const double* A, const double* B, double* C) {   // C = A*B, C must not alias
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            double s = A[i * 3 + 0] * B[0 * 3 + j];
            s = s + A[i * 3 + 1] * B[1 * 3 + j];
            s = s + A[i * 3 + 2] * B[2 * 3 + j];
            C[i * 3 + j] = s;
        }
}

// returns false (and zeros) when det == 0, like cv::invert
VSTAB_HD bool invert3(const double* a, double* t) {
    double d = a[0] * (a[4] * a[8] - a[5] * a[7]) - a[1] * (a[3] * a[8] - a[5] * a[6]) +
               a[2] * (a[3] * a[7] - a[4] * a[6]);
    if (d == 0.0) {
        for (int i = 0; i < 9; ++i) t[i] = 0.0;
        return false;
    }
    d = 1.0 / d;
    t[0] = (a[4] * a[8] - a[5] * a[7]) * d;
    t[1] = (a[2] * a[7] - a[1] * a[8]) * d;
    t[2] = (a[1] * a[5] - a[2] * a[4]) * d;
    t[3] = (a[5] * a[6] - a[3] * a[8]) * d;
    t[4] = (a[0] * a[8] - a[2] * a[6]) * d;
    t[5] = (a[2] * a[3] - a[0] * a[5]) * d;
    t[6] = (a[3] * a[7] - a[4] * a[6]) * d;
    t[7] = (a[1] * a[6] - a[0] * a[7]) * d;
    t[8] = (a[0] * a[4] - a[1] * a[3]) * d;
    return true;
}

VSTAB_HD bool finite9(const double* H) {
    for (int i = 0; i < 9; ++i)
        if (!isfinite(H[i])) return false;
    return true;
}

VSTAB_HD bool decompose_h(const double* H, double cx, double cy, HParams* out) {
    const double eps = 1e-6;
    if (!finite9(H)) return false;
    const double h33 = H[8];
    if (fabs(h33) < eps) return false;
    double Hn[9];
    for (int i = 0; i < 9; ++i) Hn[i] = H[i] / h33;
    const double tx = Hn[2], ty = Hn[5], v0 = Hn[6], v1 = Hn[7];
    // sRK = A - t v^T
    const double m00 = Hn[0] - tx * v0, m01 = Hn[1] - tx * v1;
    const double m10 = Hn[3] - ty * v0, m11 = Hn[4] - ty * v1;
    if (!(isfinite(m00) && isfinite(m01) && isfinite(m10) && isfinite(m11))) return false;
    const double det = m00 * m11 - m01 * m10;
    if (isnan(det) || isinf(det) || det < 0 || fabs(det) < eps) return false;
    const double s = sqrt(det);
    const double a00 = m00 / s, a01 = m01 / s, a10 = m10 / s, a11 = m11 / s;
    // qrDecomposition2x2 (Gram-Schmidt); every throw of the reference -> false
    if (fabs(a00 * a11 - a01 * a10) < eps) return false;
    const double n1 = sqrt(a00 * a00 + a10 * a10);
    if (n1 < eps) return false;
    const double q1x = a00 / n1, q1y = a10 / n1;
    const double r12 = a01 * q1x + a11 * q1y;
    const double u2x = a01 - r12 * q1x, u2y = a11 - r12 * q1y;
    const double n2 = sqrt(u2x * u2x + u2y * u2y);
    if (n2 < eps) return false;
    const double q2x = u2x / n2, q2y = u2y / n2;
    // Q = [q1 q2], R = [n1 r12; 0 n2]; self checks |A - QR|inf, |Q^T Q - I|inf <= eps
    {
        const double e00 = a00 - (q1x * n1), e01 = a01 - (q1x * r12 + q2x * n2);
        const double e10 = a10 - (q1y * n1), e11 = a11 - (q1y * r12 + q2y * n2);
        const double r0 = fabs(e00) + fabs(e01), r1 = fabs(e10) + fabs(e11);
        if ((r0 > r1 ? r0 : r1) > eps) return false;
        const double g00 = q1x * q1x + q1y * q1y - 1.0, g01 = q1x * q2x + q1y * q2y;
        const double g11 = q2x * q2x + q2y * q2y - 1.0;
        const double s0 = fabs(g00) + fabs(g01), s1 = fabs(g01) + fabs(g11);
        if ((s0 > s1 ? s0 : s1) > eps) return false;
    }
    if (!(isfinite(q1x) && isfinite(q1y) && isfinite(q2x) && isfinite(q2y) && isfinite(n1) &&
          isfinite(r12) && isfinite(n2)))
        return false;
    const double detR = q1x * q2y - q2x * q1y;
    if (fabs(detR - 1.0) > eps) return false;
    const double cos_t = (q1x + q2y) / 2, sin_t = (q1y - q2x) / 2;
    const double theta = atan2(sin_t, cos_t);
    // t_shift = (I - s R) c
    const double sx = (1.0 - s * q1x) * cx + (0.0 - s * q2x) * cy;
    const double sy = (0.0 - s * q1y) * cx + (1.0 - s * q2y) * cy;
    out->s = s;
    out->theta = theta;
    out->k = n1;
    out->delta = r12;
    out->t[0] = tx - sx;
    out->t[1] = ty - sy;
    out->v[0] = v0;
    out->v[1] = v1;
    return true;
}

VSTAB_HD void compose_h(const HParams* p, double cx, double cy, double* H) {
    const double c = cos(p->theta), sn = sin(p->theta);
    const double r00 = c, r01 = -sn, r10 = sn, r11 = c;
    const double k00 = p->k, k01 = p->delta, k11 = 1 / p->k;
    const double sx = (1.0 - p->s * r00) * cx + (0.0 - p->s * r01) * cy;
    const double sy = (0.0 - p->s * r10) * cx + (1.0 - p->s * r11) * cy;
    const double tx = p->t[0] + sx, ty = p->t[1] + sy;
    // A = s R K + t v^T
    const double sr00 = p->s * r00, sr01 = p->s * r01, sr10 = p->s * r10, sr11 = p->s * r11;
    H[0] = (sr00 * k00 + sr01 * 0.0) + tx * p->v[0];
    H[1] = (sr00 * k01 + sr01 * k11) + tx * p->v[1];
    H[3] = (sr10 * k00 + sr11 * 0.0) + ty * p->v[0];
    H[4] = (sr10 * k01 + sr11 * k11) + ty * p->v[1];
    H[2] = tx;
    H[5] = ty;
    H[6] = p->v[0];
    H[7] = p->v[1];
    H[8] = 1.0;
}

// ---- auto-crop (K16, vstab_set_crop; semantics in include/vstab.h) ---------------------------------------------------
// Zoom about the centre c0 of a rows x cols frame that keeps the warp by H from showing any point outside the pixel-centre
// rectangle S = [0, cols-1] x [0, rows-1]: the least z >= 1 with Z(z)^-1(S) inside Q = H(S), clamped to max_zoom.
// Q is convex when w > 0 at every corner of S; for each edge (a, b) of Q, oriented so that its inside is on the left, the
// corner q of S shrunk towards c0 by t stays inside while s0 + t * s1 >= 0.  Operation order is fixed (the restatement in
// tests/crop_ref.py follows it; crop.cu is built without FMA contraction).
VSTAB_HD double crop_need(const double* H, int rows, int cols, double max_zoom) {
    if (!finite9(H)) return max_zoom;
    const double xs[4] = {0.0, cols - 1.0, cols - 1.0, 0.0};
    const double ys[4] = {0.0, 0.0, rows - 1.0, rows - 1.0};
    double qx[4], qy[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const double w = H[6] * xs[k] + H[7] * ys[k] + H[8];
        if (!(w > 0.0)) return max_zoom;
        qx[k] = (H[0] * xs[k] + H[1] * ys[k] + H[2]) / w;
        qy[k] = (H[3] * xs[k] + H[4] * ys[k] + H[5]) / w;
    }
    double area2 = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) area2 = area2 + (qx[k] * qy[(k + 1) & 3] - qx[(k + 1) & 3] * qy[k]);
    const double sg = area2 > 0.0 ? 1.0 : -1.0;         // edge k runs Q[k] -> Q[k+1]; sg puts its inside on the left
    const double cx = (cols - 1.0) * 0.5, cy = (rows - 1.0) * 0.5;
    double t = 1.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const double ex = qx[(k + 1) & 3] - qx[k], ey = qy[(k + 1) & 3] - qy[k];
        const double s0 = sg * (ex * (cy - qy[k]) - ey * (cx - qx[k]));
        if (!(s0 > 0.0)) return max_zoom;               // the centre is not inside Q
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double s1 = sg * (ex * (ys[j] - cy) - ey * (xs[j] - cx));
            if (s1 < 0.0) {
                const double b = s0 / -s1;
                if (b < t) t = b;
            }
        }
    }
    const double z = 1.0 / t;
    return z < 1.0 ? 1.0 : (z > max_zoom ? max_zoom : z);
}

// Hc = Z(z) * H, Z(z) = [[z, 0, (1-z) c0x], [0, z, (1-z) c0y], [0, 0, 1]]
VSTAB_HD void crop_apply(double z, const double* H, int rows, int cols, double* Hc) {
    const double cx = (cols - 1.0) * 0.5, cy = (rows - 1.0) * 0.5;
    const double Z[9] = {z, 0.0, (1.0 - z) * cx, 0.0, z, (1.0 - z) * cy, 0.0, 0.0, 1.0};
    matmul3(Z, H, Hc);
}

}  // namespace vstabk
