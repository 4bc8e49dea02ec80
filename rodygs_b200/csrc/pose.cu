// Test-time pose refinement of one held-out camera: the two small kernels that, with rdg_preprocess_fwd / rdg_bin_tiles /
// rdg_blend_fwd / rdg_blend_bwd / rdg_preprocess_bwd, make one iteration of the reference's PoseOptimizer (render the static
// model, L2 photometric loss, backward, Adam step on one LearnableCamera) device-resident, so that the whole loop is
// replays of one CUDA graph with no host read.  Definitions: INTEGRATION.md "Refining held-out camera poses".
//
// Pose parameters (q, T): q = (r, x, y, z) the camera-to-world rotation (any norm; it is normalised here), T the
// camera-to-world translation.  R = rot(q / |q|),  V = [[R^T, -R^T T], [0, 0, 0, 1]].  In glm storage (the 16 floats of
// V^T row-major) the rotation block reads R row-major: V_glm[4 k + r] = V[r][k] = R[k][r] for r, k < 3.
#include <math.h>
#include "common.cuh"

#define PL_THREADS 256
#define PL_MAX_CTAS 592            // 4 per SM: enough to stream the image at full bandwidth

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
__device__ void pose_write_view(const float* prm, float* __restrict__ vm) {
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

// One warp.  Lanes 0..15 own one float of dL/dV (read, then zeroed for the next iteration's rdg_preprocess_bwd), lanes 0..6
// one Adam parameter; lane 0 chains dL/dV to dL/d(q, T) in between.
__global__ void __launch_bounds__(32) pose_adam_kernel(RdgPoseAdam a, int update) {
    __shared__ float gv[16];
    __shared__ float g7[7];
    __shared__ int apply;
    const int lane = threadIdx.x;
    if (!update) {
        if (lane == 0) pose_write_view(a.param, a.viewmatrix);
        return;
    }
    if (lane < 16) {
        gv[lane] = a.dL_dV[lane];
        a.dL_dV[lane] = 0.f;
    }
    __syncwarp();
    if (lane == 0) {
        const int step = *a.step;
        const bool overflow = a.num_rendered != nullptr && a.num_rendered[1] != 0u;
        if (overflow && a.overflow) {
            a.overflow[0] = 1u;
            a.overflow[1] = a.num_rendered[0];
        }
        apply = !overflow && step < a.max_steps;
        float qn[4], R[9];
        const float inv = pose_rot(a.param, qn, R);
        const float* T = a.param + 4;
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
    __syncwarp();
    if (lane < 7 && a.grad) a.grad[lane] = g7[lane];
    if (apply && lane < 7) {
        // torch.optim.Adam (no weight decay, no amsgrad): scalars in double as torch takes them on the host, each rounded to
        // float where the float32 tensor op consumes it
        const int t = *a.step + 1;
        const double bc1 = 1.0 - pow(a.beta1, (double)t);
        const double bc2_sqrt = sqrt(1.0 - pow(a.beta2, (double)t));
        const float g = g7[lane];
        float m = a.exp_avg[lane], v = a.exp_avg_sq[lane];
        m = m + (float)(1.0 - a.beta1) * (g - m);                     // exp_avg.lerp_(grad, 1 - beta1)
        v = v * (float)a.beta2 + (float)(1.0 - a.beta2) * g * g;      // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
        const float denom = sqrtf(v) / (float)bc2_sqrt + (float)a.eps;
        a.param[lane] = a.param[lane] + (float)(-(a.lr / bc1)) * (m / denom);
        a.exp_avg[lane] = m;
        a.exp_avg_sq[lane] = v;
    }
    __syncwarp();
    if (apply && lane == 0) {
        *a.step = *a.step + 1;
        pose_write_view(a.param, a.viewmatrix);
    }
}

extern "C" int rdg_pose_adam(const RdgPoseAdam* args, int32_t update, void* stream) {
    RDG_CHECK_ARG(args, "args is NULL");
    RDG_CHECK_ARG(args->param, "param is NULL");
    RDG_CHECK_ARG(args->viewmatrix, "viewmatrix is NULL");
    RDG_CHECK_ARG(update == 0 || update == 1, "update must be 0 or 1");
    if (update) {
        RDG_CHECK_ARG(args->exp_avg, "exp_avg is NULL");
        RDG_CHECK_ARG(args->exp_avg_sq, "exp_avg_sq is NULL");
        RDG_CHECK_ARG(args->step, "step is NULL");
        RDG_CHECK_ARG(args->dL_dV, "dL_dV is NULL");
        RDG_CHECK_ARG(args->max_steps >= 1, "max_steps must be >= 1");
        RDG_CHECK_ARG(args->lr > 0.0 && isfinite(args->lr), "lr must be a finite value > 0");
        RDG_CHECK_ARG(args->beta1 >= 0.0 && args->beta1 < 1.0, "beta1 must be in [0, 1)");
        RDG_CHECK_ARG(args->beta2 >= 0.0 && args->beta2 < 1.0, "beta2 must be in [0, 1)");
        RDG_CHECK_ARG(args->eps >= 0.0 && isfinite(args->eps), "eps must be a finite value >= 0");
        RDG_CHECK_ARG(!args->num_rendered || args->overflow, "overflow is NULL (required with num_rendered)");
    }
    pose_adam_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(*args, update);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}

// ---- L2 photometric loss ------------------------------------------------------------------------------------------------

static int l2_ctas(int64_t n) {
    const int64_t want = (n + PL_THREADS * 8 - 1) / (PL_THREADS * 8);
    return (int)(want < PL_MAX_CTAS ? (want < 1 ? 1 : want) : PL_MAX_CTAS);
}

// dL/dpred = 2 (pred - gt) / n; part[blockIdx.x] = this CTA's sum of (pred - gt)^2 (float64)
__global__ void __launch_bounds__(PL_THREADS) l2_loss_kernel(const float* __restrict__ pred, const float* __restrict__ gt, int64_t n,
                                                             float scale, float* __restrict__ dpred, double* __restrict__ part) {
    __shared__ double red[PL_THREADS / 32];
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * PL_THREADS + threadIdx.x; i < n; i += (int64_t)gridDim.x * PL_THREADS) {
        const float d = pred[i] - gt[i];
        dpred[i] = scale * d;
        acc += (double)d * (double)d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < PL_THREADS / 32; ++w) t += red[w];
        part[blockIdx.x] = t;
    }
}

// fixed-order sum of the per-CTA partials -> history[*step] (when *step < max_steps)
__global__ void __launch_bounds__(PL_THREADS) l2_finalize_kernel(const double* __restrict__ part, int count, double inv_n,
                                                                 const int32_t* __restrict__ step, int32_t max_steps,
                                                                 float* __restrict__ history) {
    __shared__ double sh[PL_THREADS];
    double t = 0.0;
    for (int i = threadIdx.x; i < count; i += PL_THREADS) t += part[i];
    sh[threadIdx.x] = t;
    __syncthreads();
    for (int s = PL_THREADS / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const int k = *step;
        if (k >= 0 && k < max_steps) history[k] = (float)(sh[0] * inv_n);
    }
}

static int l2_check_sizes(const char* fn, int32_t channels, int32_t height, int32_t width) {
    if (channels < 1) { rdg_set_error("%s: channels must be >= 1 (got %d)", fn, channels); return RDG_E_ARG; }
    if (height < 1) { rdg_set_error("%s: height must be >= 1 (got %d)", fn, height); return RDG_E_ARG; }
    if (width < 1) { rdg_set_error("%s: width must be >= 1 (got %d)", fn, width); return RDG_E_ARG; }
    return RDG_OK;
}

extern "C" int64_t rdg_l2_loss_workspace_bytes(int32_t channels, int32_t height, int32_t width) {
    const int rc = l2_check_sizes(__func__, channels, height, width);
    if (rc != RDG_OK) return rc;
    return rdg_align_up((int64_t)l2_ctas((int64_t)channels * height * width) * (int64_t)sizeof(double), 256);
}

extern "C" int rdg_l2_loss(const float* pred, const float* gt, int32_t channels, int32_t height, int32_t width,
                           const int32_t* step, int32_t max_steps, float* history, float* dL_dpred, void* workspace,
                           int64_t workspace_bytes, void* stream) {
    RDG_CHECK_ARG(pred, "pred is NULL");
    RDG_CHECK_ARG(gt, "gt is NULL");
    RDG_CHECK_ARG(step, "step is NULL");
    RDG_CHECK_ARG(history, "history is NULL");
    RDG_CHECK_ARG(dL_dpred, "dL_dpred is NULL");
    RDG_CHECK_ARG(workspace, "workspace is NULL");
    const int rc = l2_check_sizes(__func__, channels, height, width);
    if (rc != RDG_OK) return rc;
    RDG_CHECK_ARG(max_steps >= 1, "max_steps must be >= 1");
    const int64_t n = (int64_t)channels * height * width;
    const int ctas = l2_ctas(n);
    RDG_CHECK_ARG(workspace_bytes >= rdg_align_up((int64_t)ctas * (int64_t)sizeof(double), 256),
                  "workspace_bytes is smaller than rdg_l2_loss_workspace_bytes()");
    RDG_CHECK_ARG(((uintptr_t)workspace & 7) == 0, "workspace must be 8-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    double* part = (double*)workspace;
    l2_loss_kernel<<<ctas, PL_THREADS, 0, s>>>(pred, gt, n, (float)(2.0 / (double)n), dL_dpred, part);
    RDG_CHECK_LAUNCH();
    l2_finalize_kernel<<<1, PL_THREADS, 0, s>>>(part, ctas, 1.0 / (double)n, step, max_steps, history);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(2);
    return RDG_OK;
}
