// odom_math.cuh -- the estimation gate of LidarOdometry::evaluateEstimation (src/lidar_odometry.cpp:267-296) on row-major
// float 4x4 matrices, shared by the host call (bshot_evaluate_estimation, capi.cu) and the device step (odometry.cu).  Only
// IEEE +, -, *, /: the device side is compiled with -fmad=false, so both sides give the same bits.  acosf is the one
// exception (device acosf and glibc's may differ in the last bits).
#pragma once
#include <math.h>

namespace bshot {

// general 4x4 inverse by cofactors in float (Matrix4f::inverse(), src/lidar_odometry.cpp:269)
__host__ __device__ inline void inverse4x4(const float* m, float* o) {
    float inv[16];
    inv[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
    inv[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
    inv[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
    inv[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
    inv[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
    inv[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
    inv[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
    inv[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
    inv[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
    inv[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
    inv[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
    inv[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
    inv[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
    inv[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
    inv[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
    inv[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
    const float det = m[0] * inv[0] + m[1] * inv[4] + m[2] * inv[8] + m[3] * inv[12];
    const float id = 1.0f / det;
    for (int e = 0; e < 16; ++e) o[e] = inv[e] * id;
}

__host__ __device__ inline void mul4x4(const float* a, const float* b, float* o) {
    float r[16];
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) r[4 * i + j] = ((a[4 * i] * b[j] + a[4 * i + 1] * b[4 + j]) + a[4 * i + 2] * b[8 + j]) + a[4 * i + 3] * b[12 + j];
    for (int e = 0; e < 16; ++e) o[e] = r[e];
}

// rigid inverse [R^T | -R^T t] of a row-major [R|t; 0 0 0 1]: -(((r0i t0 + r1i t1) + r2i t2)) per row i (loop closure's T_rel)
__host__ __device__ inline void rigid_inverse4x4(const float* m, float* o) {
    float r[16];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) r[4 * i + j] = m[4 * j + i];
        r[4 * i + 3] = -((m[i] * m[3] + m[4 + i] * m[7]) + m[8 + i] * m[11]);
        r[12 + i] = 0.0f;
    }
    r[15] = 1.0f;
    for (int e = 0; e < 16; ++e) o[e] = r[e];
}

// T_ij = T_ref^-1 * T_ransac; heading change acos(T_ij(1,1)), translation |t_ij|; returns true when the estimate is rejected
// (more than 10 degrees, more than 1200 mm or fewer than 15 correspondences, :281)
__host__ __device__ inline bool estimation_gate(const float* T_ransac, const float* T_ref, int n_correspondences, float* h_diff, float* t_diff) {
    float Ti_inv[16], Tij[16];
    inverse4x4(T_ref, Ti_inv);
    mul4x4(Ti_inv, T_ransac, Tij);                                   // T_ij = T_i.inverse() * T_j (:269)
    *h_diff = acosf(Tij[5]);                                         // heading (0,1,0): heading^T R heading = R(1,1) (:271-272)
    *t_diff = sqrtf((Tij[3] * Tij[3] + Tij[7] * Tij[7]) + Tij[11] * Tij[11]);
    return (double)(*h_diff * 180) / M_PI > 10 || *t_diff > 1200 || n_correspondences < 15;
}

}  // namespace bshot
