// Pose arithmetic shared by rdg_pose_adam (one held-out camera) and rdg_camera_grad / rdg_camera_adam (the table of training
// cameras), so that both optimise exactly the same V(q, T).
//
// Pose parameters (q, T): q = (r, x, y, z) the camera-to-world rotation (any norm; it is normalised here), T the
// camera-to-world translation.  R = rot(q / |q|),  V = [[R^T, -R^T T], [0, 0, 0, 1]].  In glm storage (the 16 floats of
// V^T row-major) the rotation block reads R row-major: V_glm[4 k + r] = V[r][k] = R[k][r] for r, k < 3.
#pragma once
#include <math.h>

// R (row-major) of the normalised quaternion; qn receives q / |q|, the return value is 1 / |q|.
__device__ __forceinline__ float pose_rot(const float* q, float* qn, float* R) {
    const float inv = 1.0f / sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    const float r = q[0] * inv, x = q[1] * inv, y = q[2] * inv, z = q[3] * inv;
    qn[0] = r; qn[1] = x; qn[2] = y; qn[3] = z;
    R[0] = 1.f - 2.f * (y * y + z * z); R[1] = 2.f * (x * y - r * z);       R[2] = 2.f * (x * z + r * y);
    R[3] = 2.f * (x * y + r * z);       R[4] = 1.f - 2.f * (x * x + z * z); R[5] = 2.f * (y * z - r * x);
    R[6] = 2.f * (x * z - r * y);       R[7] = 2.f * (y * z + r * x);       R[8] = 1.f - 2.f * (x * x + y * y);
    return inv;
}

// V(q, T) in glm storage (16 floats)
static __device__ void pose_write_view(const float* prm, float* __restrict__ vm) {
    float qn[4], R[9];
    pose_rot(prm, qn, R);
    const float* T = prm + 4;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
#pragma unroll
        for (int r = 0; r < 3; ++r) vm[4 * k + r] = R[3 * k + r];
        vm[4 * k + 3] = 0.f;
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) vm[12 + r] = -(R[r] * T[0] + R[3 + r] * T[1] + R[6 + r] * T[2]);
    vm[15] = 1.f;
}

// dL/dV (glm storage, 16 floats) -> dL/d(q, T) (7 floats) at the pose prm, through the normalised quaternion
__device__ __forceinline__ void pose_pullback(const float* prm, const float* gv, float* g7) {
    float qn[4], R[9];
    const float inv = pose_rot(prm, qn, R);
    const float* T = prm + 4;
    // V[r][k] = R[k][r], V[r][3] = -sum_k R[k][r] T[k]; dL/dV[r][k] = gv[4 k + r]
    float dR[9];
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int r = 0; r < 3; ++r) dR[3 * k + r] = gv[4 * k + r] - T[k] * gv[12 + r];
#pragma unroll
    for (int k = 0; k < 3; ++k) g7[4 + k] = -(R[3 * k] * gv[12] + R[3 * k + 1] * gv[13] + R[3 * k + 2] * gv[14]);
    const float r = qn[0], x = qn[1], y = qn[2], z = qn[3];
    float dq[4];
    dq[0] = 2.f * (-z * dR[1] + y * dR[2] + z * dR[3] - x * dR[5] - y * dR[6] + x * dR[7]);
    dq[1] = 2.f * (y * dR[1] + z * dR[2] + y * dR[3] - 2.f * x * dR[4] - r * dR[5] + z * dR[6] + r * dR[7] - 2.f * x * dR[8]);
    dq[2] = 2.f * (-2.f * y * dR[0] + x * dR[1] + r * dR[2] + x * dR[3] + z * dR[5] - r * dR[6] + z * dR[7] - 2.f * y * dR[8]);
    dq[3] = 2.f * (-2.f * z * dR[0] - r * dR[1] + x * dR[2] + r * dR[3] - 2.f * z * dR[4] + y * dR[5] + x * dR[6] + y * dR[7]);
    // through q / |q|: (I - qn qn^T) / |q|
    const float dot = r * dq[0] + x * dq[1] + y * dq[2] + z * dq[3];
#pragma unroll
    for (int k = 0; k < 4; ++k) g7[k] = (dq[k] - qn[k] * dot) * inv;
}

// One element of torch.optim.Adam (no weight decay, no amsgrad) at step t >= 1: scalars in double as torch takes them on
// the host, each rounded to float where the float32 tensor op consumes it
__device__ __forceinline__ void pose_adam_elem(float& p, float g, float& m, float& v, int t, double lr, double beta1, double beta2,
                                               double eps) {
    const double bc1 = 1.0 - pow(beta1, (double)t);
    const double bc2_sqrt = sqrt(1.0 - pow(beta2, (double)t));
    m = m + (float)(1.0 - beta1) * (g - m);                     // exp_avg.lerp_(grad, 1 - beta1)
    v = v * (float)beta2 + (float)(1.0 - beta2) * g * g;        // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    const float denom = sqrtf(v) / (float)bc2_sqrt + (float)eps;
    p = p + (float)(-(lr / bc1)) * (m / denom);
}
