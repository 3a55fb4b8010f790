// eigh3.cuh -- fp64 eigen-decomposition of a symmetric 3x3 on the device, shared by the SHOT local reference frame
// (shot.cu) and the ISS saliency pass (iss.cu).
#pragma once
#include "common.cuh"

namespace bshot {

// cyclic Jacobi eigen-decomposition of a symmetric 3x3 (fp64); ascending eigenvalues, columns of V
__device__ inline void eigh3_jacobi(const double m[6] /*xx,xy,xz,yy,yz,zz*/, double w[3], double V[3][3]) {
    double a[3][3] = {{m[0], m[1], m[2]}, {m[1], m[3], m[4]}, {m[2], m[4], m[5]}};
    double v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int sweep = 0; sweep < 32; ++sweep) {
        const double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2];
        const double diag = a[0][0] * a[0][0] + a[1][1] * a[1][1] + a[2][2] * a[2][2];
        if (!(off > 1e-40 * diag)) break;
#pragma unroll
        for (int p = 0; p < 2; ++p) {
#pragma unroll
            for (int q = p + 1; q < 3; ++q) {
                const double apq = a[p][q];
                if (apq == 0.0) continue;
                const double theta = (a[q][q] - a[p][p]) / (2.0 * apq);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const double akp = a[k][p], akq = a[k][q];
                    a[k][p] = cs * akp - sn * akq;
                    a[k][q] = sn * akp + cs * akq;
                }
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const double apk = a[p][k], aqk = a[q][k];
                    a[p][k] = cs * apk - sn * aqk;
                    a[q][k] = sn * apk + cs * aqk;
                }
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const double vkp = v[k][p], vkq = v[k][q];
                    v[k][p] = cs * vkp - sn * vkq;
                    v[k][q] = sn * vkp + cs * vkq;
                }
            }
        }
    }
    int o0 = 0, o1 = 1, o2 = 2;
    double d0 = a[0][0], d1 = a[1][1], d2 = a[2][2];
    if (d0 > d1) { double t = d0; d0 = d1; d1 = t; int ti = o0; o0 = o1; o1 = ti; }
    if (d1 > d2) { double t = d1; d1 = d2; d2 = t; int ti = o1; o1 = o2; o2 = ti; }
    if (d0 > d1) { double t = d0; d0 = d1; d1 = t; int ti = o0; o0 = o1; o1 = ti; }
    w[0] = d0; w[1] = d1; w[2] = d2;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        V[r][0] = (o0 == 0) ? v[r][0] : (o0 == 1 ? v[r][1] : v[r][2]);
        V[r][1] = (o1 == 0) ? v[r][0] : (o1 == 1 ? v[r][1] : v[r][2]);
        V[r][2] = (o2 == 0) ? v[r][0] : (o2 == 1 ? v[r][1] : v[r][2]);
    }
}

}  // namespace bshot
