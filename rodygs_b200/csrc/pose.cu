// Test-time pose refinement of one held-out camera: the two small kernels that, with rdg_preprocess_fwd / rdg_bin_tiles /
// rdg_blend_fwd / rdg_blend_bwd / rdg_preprocess_bwd, make one iteration of the reference's PoseOptimizer (render the static
// model, L2 photometric loss, backward, Adam step on one LearnableCamera) device-resident, so that the whole loop is
// replays of one CUDA graph with no host read.  Definitions: INTEGRATION.md "Refining held-out camera poses".
//
// The pose arithmetic (V(q, T), dL/dV -> dL/d(q, T), the Adam element) is in pose.cuh, shared with the camera table below.
#include <math.h>
#include "common.cuh"
#include "pose.cuh"

#define PL_THREADS 256
#define PL_MAX_CTAS 592            // 4 per SM: enough to stream the image at full bandwidth

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
        pose_pullback(a.param, gv, g7);
    }
    __syncwarp();
    if (lane < 7 && a.grad) a.grad[lane] = g7[lane];
    if (apply && lane < 7) {
        float p = a.param[lane], m = a.exp_avg[lane], v = a.exp_avg_sq[lane];
        pose_adam_elem(p, g7[lane], m, v, *a.step + 1, a.lr, a.beta1, a.beta2, a.eps);
        a.param[lane] = p;
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

// ---- the table of training cameras (INTEGRATION.md "Learning the training cameras") --------------------------------------
// C is at most a few thousand rows of 7 floats: each launch below is one thread per camera and takes microseconds, so
// none of them is tuned.

#define CAM_THREADS 128

// One thread per camera: its row of dL/d(q, T) is the slot-order sum of the pulled-back dL/dV of every slot naming it (no
// atomics, so the result is bit-identical from run to run; a row no slot names is 0).  Thread 0 also scans the indices and
// writes 1 + the first slot whose camera lies outside [0, C) into *error, or 0; such a slot adds to no row.
__global__ void __launch_bounds__(CAM_THREADS) camera_grad_kernel(int n_slots, const int32_t* __restrict__ cam_idx,
                                                                  const float* __restrict__ dV, const float* __restrict__ param,
                                                                  int C, float* __restrict__ grad, int32_t* __restrict__ error) {
    const int c = blockIdx.x * CAM_THREADS + threadIdx.x;
    if (c == 0) {
        int bad = 0;
        for (int s = 0; s < n_slots && !bad; ++s)
            if (cam_idx[s] < 0 || cam_idx[s] >= C) bad = s + 1;
        *error = bad;
    }
    if (c >= C) return;
    float prm[7], acc[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) prm[k] = param[7 * c + k];
    bool have = false;
    for (int s = 0; s < n_slots; ++s) {
        if (cam_idx[s] != c) continue;
        float gv[16], g7[7];
#pragma unroll
        for (int k = 0; k < 16; ++k) gv[k] = dV[16 * s + k];
        pose_pullback(prm, gv, g7);
        // the first term is taken as it is (0 + x would turn a -0 into +0): one slot gives rdg_pose_adam's bits
#pragma unroll
        for (int k = 0; k < 7; ++k) acc[k] = have ? acc[k] + g7[k] : g7[k];
        have = true;
    }
#pragma unroll
    for (int k = 0; k < 7; ++k) grad[7 * c + k] = have ? acc[k] : 0.f;
}

// One thread per camera: one Adam step of all 7 parameters (q with lr_q, T with lr_T), then V(q, T) of the new pose
__global__ void __launch_bounds__(CAM_THREADS) camera_adam_kernel(float* __restrict__ param, const float* __restrict__ grad,
                                                                  float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq, int C,
                                                                  int step, double lr_q, double lr_T, double beta1, double beta2,
                                                                  double eps, float grad_scale, float* __restrict__ viewmats) {
    const int c = blockIdx.x * CAM_THREADS + threadIdx.x;
    if (c >= C) return;
    float prm[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        const int i = 7 * c + k;
        float p = param[i], m = exp_avg[i], v = exp_avg_sq[i];
        pose_adam_elem(p, grad[i] * grad_scale, m, v, step, k < 4 ? lr_q : lr_T, beta1, beta2, eps);
        param[i] = prm[k] = p;
        exp_avg[i] = m;
        exp_avg_sq[i] = v;
    }
    pose_write_view(prm, viewmats + 16 * c);
}

__global__ void __launch_bounds__(CAM_THREADS) camera_views_kernel(const float* __restrict__ param, int C,
                                                                   float* __restrict__ viewmats) {
    const int c = blockIdx.x * CAM_THREADS + threadIdx.x;
    if (c < C) pose_write_view(param + 7 * c, viewmats + 16 * c);
}

extern "C" int rdg_camera_grad(int32_t n_slots, const int32_t* cam_idx, const float* dL_dV_slots, const float* param, int32_t C,
                               float* grad, int32_t* error, void* stream) {
    RDG_CHECK_ARG(cam_idx, "cam_idx is NULL");
    RDG_CHECK_ARG(dL_dV_slots, "dL_dV_slots is NULL");
    RDG_CHECK_ARG(param, "param is NULL");
    RDG_CHECK_ARG(grad, "grad is NULL");
    RDG_CHECK_ARG(error, "error is NULL");
    RDG_CHECK_ARG(n_slots >= 0, "n_slots must be >= 0");
    RDG_CHECK_ARG(C >= 1, "C must be >= 1");
    camera_grad_kernel<<<rdg_div_up(C, CAM_THREADS), CAM_THREADS, 0, (cudaStream_t)stream>>>(n_slots, cam_idx, dL_dV_slots,
                                                                                            param, C, grad, error);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}

extern "C" int rdg_camera_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int32_t C, int32_t step,
                               double lr_q, double lr_T, double beta1, double beta2, double eps, float grad_scale, float* viewmats,
                               void* stream) {
    RDG_CHECK_ARG(param, "param is NULL");
    RDG_CHECK_ARG(grad, "grad is NULL");
    RDG_CHECK_ARG(exp_avg, "exp_avg is NULL");
    RDG_CHECK_ARG(exp_avg_sq, "exp_avg_sq is NULL");
    RDG_CHECK_ARG(viewmats, "viewmats is NULL");
    RDG_CHECK_ARG(C >= 1, "C must be >= 1");
    RDG_CHECK_ARG(step >= 1, "step must be >= 1");
    RDG_CHECK_ARG(lr_q >= 0.0 && isfinite(lr_q), "lr_q must be a finite value >= 0");
    RDG_CHECK_ARG(lr_T >= 0.0 && isfinite(lr_T), "lr_T must be a finite value >= 0");
    RDG_CHECK_ARG(beta1 >= 0.0 && beta1 < 1.0, "beta1 must be in [0, 1)");
    RDG_CHECK_ARG(beta2 >= 0.0 && beta2 < 1.0, "beta2 must be in [0, 1)");
    RDG_CHECK_ARG(eps >= 0.0 && isfinite(eps), "eps must be a finite value >= 0");
    RDG_CHECK_ARG(isfinite(grad_scale), "grad_scale must be finite");
    camera_adam_kernel<<<rdg_div_up(C, CAM_THREADS), CAM_THREADS, 0, (cudaStream_t)stream>>>(
        param, grad, exp_avg, exp_avg_sq, C, step, lr_q, lr_T, beta1, beta2, eps, grad_scale, viewmats);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}

extern "C" int rdg_camera_views(const float* param, int32_t C, float* viewmats, void* stream) {
    RDG_CHECK_ARG(param, "param is NULL");
    RDG_CHECK_ARG(viewmats, "viewmats is NULL");
    RDG_CHECK_ARG(C >= 1, "C must be >= 1");
    camera_views_kernel<<<rdg_div_up(C, CAM_THREADS), CAM_THREADS, 0, (cudaStream_t)stream>>>(param, C, viewmats);
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
