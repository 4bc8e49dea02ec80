// RigidityLoss, modes "surface" and "distance_preserving" - value and gradient in one call (SURVEY.md §8 f4).
// Reference: /root/reference/src/trainer/losses.py:216-361 (every train config: K 8, both modes, freq 5),
// CharbonnierLoss(out_norm "bc") /root/reference/src/utils/loss_utils.py:235-250.
//
// The reference materialises [n, Ts, K, 3] neighbour trajectories through knn_gather + permute + broadcast
// (n = N_d / 2 sampled Gaussians, Ts = T / 4 sampled frames: 1.2 GB per temporary at BASELINE config 4) and lets
// autograd replay all of it.  Here:
//   loc      LOC[ts][p] = canon_p + c_p . B_ts[:, :3]                       one float4 per (frame, point)
//   pairs    per (ts, i): x = | LOC[ts][nn(i,k)] - LOC[ts][i] |, the Charbonnier term against the squared
//            neighbour distance the reference's `.view(-1, Ts, 1)` pairs it with (flat element f of the contiguous
//            [Ts, n, K] block goes with neighbour-distance number f / Ts - a memory reinterpretation, reproduced
//            as it is), the force W[ts][p] on both end points (16-byte vector atomics), dL/d(dist2) per pair
//   point    dL/dcanon_p = sum_ts W, dL/dc_p[b] = sum_ts W . B_ts[b]
//   basis    dL/dB_ts[b] = sum_p c_p[b] W[ts][p]  (register accumulation over 16 points per thread, one block
//            reduction per CTA), added to d_table at the sampled frames
//   space    surface term + the chain through the squared neighbour distances, on the deformed points
// Frame-major LOC / W keep one frame's slice (16 B x n = 8 MB at config 4) resident in the 126 MB L2 while the
// (ts, *) CTAs gather from it.  Bound: L2 gather bandwidth; HBM traffic ~ (2 x 32 + 16) B x n x Ts.
#include <math.h>
#include "common.cuh"

#define RG_BLOCK 256
#define RG_B 16               // basis functions (every reference config)
#define RG_KMAX 16

__device__ __forceinline__ double rg_block_sum(double v, double* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    double r = 0.0;
    if (w == 0) {
        r = l < (blockDim.x >> 5) ? sh[l] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
    }
    return r;
}

// B_ts[:, :3] of the sampled frames into shared memory: sB[ts][b][d]
__device__ __forceinline__ void load_basis(float* sB, const float* __restrict__ table, const int32_t* __restrict__ tidx,
                                           int Ts) {
    for (int e = threadIdx.x; e < Ts * RG_B * 3; e += blockDim.x) {
        const int ts = e / (RG_B * 3), rem = e % (RG_B * 3), b = rem / 3, d = rem % 3;
        sB[e] = table[((int64_t)tidx[ts] * RG_B + b) * 7 + d];
    }
    __syncthreads();
}

__device__ __forceinline__ void load_coeff(const float* __restrict__ coeff, int64_t p, float c[RG_B]) {
    const float4* src = reinterpret_cast<const float4*>(coeff + p * RG_B);
#pragma unroll
    for (int k = 0; k < RG_B / 4; ++k) {
        const float4 v = src[k];
        c[4 * k] = v.x; c[4 * k + 1] = v.y; c[4 * k + 2] = v.z; c[4 * k + 3] = v.w;
    }
}

__global__ void __launch_bounds__(RG_BLOCK) rg_loc_kernel(int64_t n, int Ts, const float* __restrict__ canon,
                                                          const float* __restrict__ coeff, const float* __restrict__ table,
                                                          const int32_t* __restrict__ tidx, float4* __restrict__ LOC) {
    extern __shared__ float sB[];
    load_basis(sB, table, tidx, Ts);
    const int64_t p = (int64_t)blockIdx.x * RG_BLOCK + threadIdx.x;
    if (p >= n) return;
    float c[RG_B];
    load_coeff(coeff, p, c);
    const float x = canon[p * 3], y = canon[p * 3 + 1], z = canon[p * 3 + 2];
    for (int ts = 0; ts < Ts; ++ts) {
        const float* Bt = sB + ts * RG_B * 3;
        float tx = 0.f, ty = 0.f, tz = 0.f;
#pragma unroll
        for (int b = 0; b < RG_B; ++b) {
            tx += c[b] * Bt[b * 3];
            ty += c[b] * Bt[b * 3 + 1];
            tz += c[b] * Bt[b * 3 + 2];
        }
        LOC[(int64_t)ts * n + p] = make_float4(x + tx, y + ty, z + tz, 0.f);
    }
}

__global__ void __launch_bounds__(RG_BLOCK) rg_pair_kernel(int64_t n, int K, int Ts, const float4* __restrict__ LOC,
                                                           const int32_t* __restrict__ nn, const float* __restrict__ dd,
                                                           float eps2, float norm, float4* __restrict__ W,
                                                           float* __restrict__ dY, double* __restrict__ sums) {
    __shared__ double sh[RG_BLOCK / 32];
    const int ts = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * RG_BLOCK + threadIdx.x;
    double lsum = 0.0;
    if (i < n) {
        const float4* L = LOC + (int64_t)ts * n;
        float4* Wt = W + (int64_t)ts * n;
        const float4 li = L[i];
        float wx = 0.f, wy = 0.f, wz = 0.f;
        int64_t f = ((int64_t)ts * n + i) * K;
        int64_t r_cur = -1;
        float gy_acc = 0.f;
        for (int k = 0; k < K; ++k, ++f) {
            const int j = nn[i * K + k];
            const float4 lj = L[j];
            const float dx = lj.x - li.x, dy = lj.y - li.y, dz = lj.z - li.z;
            const float x = sqrtf(dx * dx + dy * dy + dz * dz);
            const int64_t r = f / Ts;
            const float e = x - dd[r];
            const float term = sqrtf(e * e + eps2);
            lsum += (double)term;
            const float gx = norm * e / term;
            if (r != r_cur) {
                if (r_cur >= 0) atomicAdd(dY + r_cur, gy_acc);
                r_cur = r;
                gy_acc = 0.f;
            }
            gy_acc -= gx;
            if (x > 0.f) {                       // torch.norm backward: zero sub-gradient at 0 (k = 0 is the point itself)
                const float s = gx / x;
                const float vx = s * dx, vy = s * dy, vz = s * dz;
                wx -= vx; wy -= vy; wz -= vz;
                atomicAdd(Wt + j, make_float4(vx, vy, vz, 0.f));
            }
        }
        if (r_cur >= 0) atomicAdd(dY + r_cur, gy_acc);
        atomicAdd(Wt + i, make_float4(wx, wy, wz, 0.f));
    }
    const double tot = rg_block_sum(lsum, sh);
    if (threadIdx.x == 0) atomicAdd(sums + 1, tot);
}

__global__ void __launch_bounds__(RG_BLOCK) rg_point_kernel(int64_t n, int Ts, const float4* __restrict__ W,
                                                            const float* __restrict__ table, const int32_t* __restrict__ tidx,
                                                            float* __restrict__ d_canon, float* __restrict__ d_coeff) {
    extern __shared__ float sB[];
    load_basis(sB, table, tidx, Ts);
    const int64_t p = (int64_t)blockIdx.x * RG_BLOCK + threadIdx.x;
    if (p >= n) return;
    float dc[RG_B];
#pragma unroll
    for (int b = 0; b < RG_B; ++b) dc[b] = 0.f;
    float gx = 0.f, gy = 0.f, gz = 0.f;
    for (int ts = 0; ts < Ts; ++ts) {
        const float4 w = W[(int64_t)ts * n + p];
        const float* Bt = sB + ts * RG_B * 3;
        gx += w.x; gy += w.y; gz += w.z;
#pragma unroll
        for (int b = 0; b < RG_B; ++b) dc[b] += w.x * Bt[b * 3] + w.y * Bt[b * 3 + 1] + w.z * Bt[b * 3 + 2];
    }
    d_canon[p * 3] = gx; d_canon[p * 3 + 1] = gy; d_canon[p * 3 + 2] = gz;
    float4* dst = reinterpret_cast<float4*>(d_coeff + p * RG_B);
#pragma unroll
    for (int k = 0; k < RG_B / 4; ++k) dst[k] = make_float4(dc[4 * k], dc[4 * k + 1], dc[4 * k + 2], dc[4 * k + 3]);
}

#define RG_BASIS_PTS 16     // points per thread in the basis reduction
__global__ void __launch_bounds__(RG_BLOCK) rg_basis_kernel(int64_t n, const float4* __restrict__ W,
                                                            const float* __restrict__ coeff, const int32_t* __restrict__ tidx,
                                                            float* __restrict__ d_table) {
    __shared__ float red[RG_BLOCK / 32][RG_B * 3];
    const int ts = blockIdx.y;
    const float4* Wt = W + (int64_t)ts * n;
    float acc[RG_B * 3];
#pragma unroll
    for (int e = 0; e < RG_B * 3; ++e) acc[e] = 0.f;
    const int64_t base = (int64_t)blockIdx.x * RG_BLOCK * RG_BASIS_PTS;
    for (int it = 0; it < RG_BASIS_PTS; ++it) {
        const int64_t p = base + (int64_t)it * RG_BLOCK + threadIdx.x;
        if (p < n) {
            const float4 w = Wt[p];
            float c[RG_B];
            load_coeff(coeff, p, c);
#pragma unroll
            for (int b = 0; b < RG_B; ++b) {
                acc[b * 3] += c[b] * w.x;
                acc[b * 3 + 1] += c[b] * w.y;
                acc[b * 3 + 2] += c[b] * w.z;
            }
        }
    }
    const int wp = threadIdx.x >> 5, l = threadIdx.x & 31;
#pragma unroll
    for (int e = 0; e < RG_B * 3; ++e) {
        const float v = warp_sum(acc[e]);
        if (l == 0) red[wp][e] = v;
    }
    __syncthreads();
    if (threadIdx.x < RG_B * 3) {
        float v = 0.f;
#pragma unroll
        for (int k = 0; k < RG_BLOCK / 32; ++k) v += red[k][threadIdx.x];
        const int b = threadIdx.x / 3, d = threadIdx.x % 3;
        atomicAdd(d_table + ((int64_t)tidx[ts] * RG_B + b) * 7 + d, v);
    }
}

__global__ void __launch_bounds__(RG_BLOCK) rg_space_kernel(int64_t n, int K, const float* __restrict__ pts,
                                                            const int32_t* __restrict__ nn, const float* __restrict__ dY,
                                                            int surface, float pd_eps, float* __restrict__ d_pts,
                                                            double* __restrict__ sums) {
    __shared__ double sh[RG_BLOCK / 32];
    const int64_t i = (int64_t)blockIdx.x * RG_BLOCK + threadIdx.x;
    double lsum = 0.0;
    if (i < n) {
        const float px = pts[i * 3], py = pts[i * 3 + 1], pz = pts[i * 3 + 2];
        // p_i - mean_k p_j as the mean of the differences.  Each difference is rounded once at the scale of the difference
        // (and is exact when the two coordinates are within a factor of 2 of each other), where p_i minus the float mean
        // of the coordinates kept the sum's rounding (~ulp of the coordinates) on a value ~1e-2 of them
        float mx = 0.f, my = 0.f, mz = 0.f;
        float ax = 0.f, ay = 0.f, az = 0.f;          // gradient on the point itself
        int js[RG_KMAX];
#pragma unroll
        for (int k = 0; k < RG_KMAX; ++k)
            if (k < K) {
                const int j = nn[i * K + k];
                js[k] = j;
                mx += px - pts[(int64_t)j * 3]; my += py - pts[(int64_t)j * 3 + 1]; mz += pz - pts[(int64_t)j * 3 + 2];
            }
        float sx = 0.f, sy = 0.f, sz = 0.f;          // -(surface gradient) / K, shared by all neighbours
        if (surface) {
            const float invK = 1.0f / (float)K;
            // F.pairwise_distance(x1, x2) = || x1 - x2 + eps ||_2, eps 1e-6 (losses.py:254)
            const float dx = mx * invK + pd_eps, dy = my * invK + pd_eps, dz = mz * invK + pd_eps;
            const float s = sqrtf(dx * dx + dy * dy + dz * dz);
            lsum = (double)s;
            if (s > 0.f) {
                const float g = 1.0f / (s * (float)n);
                ax = g * dx; ay = g * dy; az = g * dz;
                sx = -ax * invK; sy = -ay * invK; sz = -az * invK;
            }
        }
#pragma unroll
        for (int k = 0; k < RG_KMAX; ++k)
            if (k < K) {
                const int64_t j = js[k];
                float gx = sx, gy = sy, gz = sz;
                if (dY) {   // dist2 = |p_i - p_j|^2 : d/dp_i = 2 (p_i - p_j) dY, d/dp_j = -that
                    const float g2 = 2.0f * dY[i * K + k];
                    const float ex = g2 * (px - pts[j * 3]), ey = g2 * (py - pts[j * 3 + 1]), ez = g2 * (pz - pts[j * 3 + 2]);
                    ax += ex; ay += ey; az += ez;
                    gx -= ex; gy -= ey; gz -= ez;
                }
                atomicAdd(d_pts + j * 3, gx);
                atomicAdd(d_pts + j * 3 + 1, gy);
                atomicAdd(d_pts + j * 3 + 2, gz);
            }
        atomicAdd(d_pts + i * 3, ax);
        atomicAdd(d_pts + i * 3 + 1, ay);
        atomicAdd(d_pts + i * 3 + 2, az);
    }
    const double tot = rg_block_sum(lsum, sh);
    if (threadIdx.x == 0 && surface) atomicAdd(sums, tot);
}

__global__ void rg_finalize_kernel(const double* __restrict__ sums, double inv_n, double norm, float* __restrict__ out) {
    out[0] = (float)(sums[0] * inv_n);
    out[1] = (float)(sums[1] * norm);
}

struct RgLayout { int64_t sums, dY, LOC, W, total; };

static RgLayout rg_layout(int64_t n, int K, int Ts) {
    RgLayout L;
    int64_t off = 0;
    L.sums = off; off += 256;
    L.dY = off; off += rdg_align_up(n * K * 4, 256);
    L.LOC = off; off += rdg_align_up((int64_t)Ts * n * 16, 256);
    L.W = off; off += rdg_align_up((int64_t)Ts * n * 16, 256);
    L.total = off;
    return L;
}

extern "C" int64_t rdg_rigidity_workspace_bytes(int64_t n, int32_t K, int32_t n_frames) {
    return (n > 0 && K > 0 && n_frames >= 0) ? rg_layout(n, K, n_frames).total : 0;
}

extern "C" int rdg_rigidity(const RdgRigidity* a, void* workspace, int64_t workspace_bytes, void* stream) {
    RDG_CHECK_ARG(a && workspace, "null argument");
    RDG_CHECK_ARG(a->n > 0 && a->K >= 1 && a->K <= RG_KMAX, "n > 0 and K in 1..16");
    RDG_CHECK_ARG(a->points && a->nn_idx && a->nn_dist2 && a->loss_parts && a->d_points, "null tensor");
    RDG_CHECK_ARG(a->mode_surface || a->mode_distance, "no mode selected");
    const int Ts = a->mode_distance ? a->n_frames : 0;
    if (a->mode_distance) {
        RDG_CHECK_ARG(a->num_basis == RG_B, "only num_basis == 16 (the reference's configs) is built");
        RDG_CHECK_ARG(a->canon && a->coeff && a->table && a->frame_indices && a->d_canon && a->d_coeff && a->d_table,
                      "distance_preserving needs canon / coeff / table / frame_indices and their gradient buffers");
        RDG_CHECK_ARG(Ts >= 1 && Ts <= 65535 && (int64_t)Ts * RG_B * 3 * 4 <= 96 * 1024, "1 <= n_frames <= 512");
        RDG_CHECK_ARG((((uintptr_t)a->coeff | (uintptr_t)a->d_coeff) & 15) == 0, "coeff / d_coeff must be 16-byte aligned");
    }
    const RgLayout L = rg_layout(a->n, a->K, Ts);
    RDG_CHECK_ARG(workspace_bytes >= L.total, "workspace too small (rdg_rigidity_workspace_bytes)");
    RDG_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    double* sums = (double*)(ws + L.sums);
    float* dY = (float*)(ws + L.dY);
    float4* LOC = (float4*)(ws + L.LOC);
    float4* W = (float4*)(ws + L.W);
    const int64_t n = a->n;
    const int pgrid = rdg_div_up(n, RG_BLOCK);
    int launches = 2;
    RDG_CUDA(cudaMemsetAsync(sums, 0, 2 * sizeof(double), st));
    RDG_CUDA(cudaMemsetAsync(a->d_points, 0, (size_t)n * 3 * 4, st));
    if (a->mode_distance) {
        const size_t smem = (size_t)Ts * RG_B * 3 * 4;
        if (smem > 48 * 1024) {
            RDG_CUDA(cudaFuncSetAttribute(rg_loc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            RDG_CUDA(cudaFuncSetAttribute(rg_point_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        }
        RDG_CUDA(cudaMemsetAsync(dY, 0, (size_t)n * a->K * 4, st));
        RDG_CUDA(cudaMemsetAsync(W, 0, (size_t)Ts * n * 16, st));
        rg_loc_kernel<<<pgrid, RG_BLOCK, smem, st>>>(n, Ts, a->canon, a->coeff, a->table, a->frame_indices, LOC);
        const double normd = 1.0 / ((double)n * a->K * Ts);
        rg_pair_kernel<<<dim3(pgrid, Ts), RG_BLOCK, 0, st>>>(n, a->K, Ts, LOC, a->nn_idx, a->nn_dist2, a->eps * a->eps,
                                                             (float)normd, W, dY, sums);
        rg_point_kernel<<<pgrid, RG_BLOCK, smem, st>>>(n, Ts, W, a->table, a->frame_indices, a->d_canon, a->d_coeff);
        rg_basis_kernel<<<dim3(rdg_div_up(n, RG_BLOCK * RG_BASIS_PTS), Ts), RG_BLOCK, 0, st>>>(n, W, a->coeff,
                                                                                                a->frame_indices, a->d_table);
        RDG_CHECK_LAUNCH();
        launches += 4;
    }
    rg_space_kernel<<<pgrid, RG_BLOCK, 0, st>>>(n, a->K, a->points, a->nn_idx, a->mode_distance ? dY : nullptr,
                                                a->mode_surface, 1e-6f, a->d_points, sums);
    RDG_CHECK_LAUNCH();
    rg_finalize_kernel<<<1, 1, 0, st>>>(sums, 1.0 / (double)n, a->mode_distance ? 1.0 / ((double)n * a->K * Ts) : 0.0,
                                        a->loss_parts);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(launches);
    return RDG_OK;
}

// ---- sample gather / scatter for the flat-buffer trainer ---------------------------------------------------------------
// The reference draws `indice` (losses.py:228-232) and indexes xyz + pred_translation, _motion_coeff with it; on the fused
// path pred_translation is never materialised (it lives inside preprocess_fwd), so the sampled rows are deformed here:
//   points_s = xyz[i] + lr * sum_b c_ib (B(t)_b - table[t_i]_b)[:3]         (src/model/rodygs_dynamic.py:122-138)
// and the backward sends d_points / d_canon / d_coeff of the sample back to the rows of the full model, to B(t) and to the
// table.  d_table is reduced per birth frame in shared memory first (T x 16 x 3 floats), flushed once per CTA; B(t)'s
// gradient is minus the sum of the table's over the frames, taken from the same accumulators.

__global__ void __launch_bounds__(RG_BLOCK) rg_sample_fwd_kernel(int64_t n, const int32_t* __restrict__ indice,
                                                                 const float* __restrict__ xyz, const float* __restrict__ coeff,
                                                                 const int32_t* __restrict__ time_ind,
                                                                 const float* __restrict__ basis_t, const float* __restrict__ table,
                                                                 float lr, float* __restrict__ points, float* __restrict__ canon,
                                                                 float* __restrict__ coeff_s) {
    const int64_t s = (int64_t)blockIdx.x * RG_BLOCK + threadIdx.x;
    if (s >= n) return;
    const int64_t i = indice[s];
    float c[RG_B];
    load_coeff(coeff, i, c);
    const float* row = table + (int64_t)time_ind[i] * RG_B * 7;
    float tx = 0.f, ty = 0.f, tz = 0.f;
#pragma unroll
    for (int b = 0; b < RG_B; ++b) {
        tx += c[b] * (basis_t[b * 7] - row[b * 7]);
        ty += c[b] * (basis_t[b * 7 + 1] - row[b * 7 + 1]);
        tz += c[b] * (basis_t[b * 7 + 2] - row[b * 7 + 2]);
    }
    const float x = xyz[i * 3], y = xyz[i * 3 + 1], z = xyz[i * 3 + 2];
    canon[s * 3] = x; canon[s * 3 + 1] = y; canon[s * 3 + 2] = z;
    points[s * 3] = x + tx * lr; points[s * 3 + 1] = y + ty * lr; points[s * 3 + 2] = z + tz * lr;
    float4* dst = reinterpret_cast<float4*>(coeff_s + s * RG_B);
#pragma unroll
    for (int k = 0; k < RG_B / 4; ++k) dst[k] = make_float4(c[4 * k], c[4 * k + 1], c[4 * k + 2], c[4 * k + 3]);
}

__global__ void __launch_bounds__(RG_BLOCK) rg_sample_bwd_kernel(int64_t n, int T, const int32_t* __restrict__ indice,
                                                                 const float* __restrict__ coeff, const int32_t* __restrict__ time_ind,
                                                                 const float* __restrict__ basis_t, const float* __restrict__ table,
                                                                 float lr, float scale, const float* __restrict__ d_points,
                                                                 const float* __restrict__ d_canon, const float* __restrict__ d_coeff_s,
                                                                 float* __restrict__ d_xyz, float* __restrict__ d_coeff,
                                                                 float* __restrict__ d_basis_t, float* __restrict__ d_table) {
    extern __shared__ float sT[];                    // [T][RG_B][3]: sum of lr * scale * c_ib * g_i over the CTA's rows
    for (int e = threadIdx.x; e < T * RG_B * 3; e += RG_BLOCK) sT[e] = 0.f;
    __syncthreads();
    for (int64_t s = (int64_t)blockIdx.x * RG_BLOCK + threadIdx.x; s < n; s += (int64_t)gridDim.x * RG_BLOCK) {
        const int64_t i = indice[s];                 // the sample has no repeated rows (random.sample): plain read-modify-write
        const float gx = d_points[s * 3], gy = d_points[s * 3 + 1], gz = d_points[s * 3 + 2];
        d_xyz[i * 3] += scale * (gx + (d_canon ? d_canon[s * 3] : 0.f));
        d_xyz[i * 3 + 1] += scale * (gy + (d_canon ? d_canon[s * 3 + 1] : 0.f));
        d_xyz[i * 3 + 2] += scale * (gz + (d_canon ? d_canon[s * 3 + 2] : 0.f));
        float c[RG_B];
        load_coeff(coeff, i, c);
        const int t = time_ind[i];
        const float* row = table + (int64_t)t * RG_B * 7;
        float* acc = sT + t * RG_B * 3;
        float4* dst = reinterpret_cast<float4*>(d_coeff + i * RG_B);
        const float4* dcs = d_coeff_s ? reinterpret_cast<const float4*>(d_coeff_s + s * RG_B) : nullptr;
        const float k = lr * scale;
#pragma unroll
        for (int q = 0; q < RG_B / 4; ++q) {
            float4 o = dst[q];
            float add[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int b = 4 * q + e;
                add[e] = k * ((basis_t[b * 7] - row[b * 7]) * gx + (basis_t[b * 7 + 1] - row[b * 7 + 1]) * gy +
                              (basis_t[b * 7 + 2] - row[b * 7 + 2]) * gz);
                atomicAdd(acc + b * 3, k * c[b] * gx);
                atomicAdd(acc + b * 3 + 1, k * c[b] * gy);
                atomicAdd(acc + b * 3 + 2, k * c[b] * gz);
            }
            if (dcs) {
                const float4 v = dcs[q];
                add[0] += scale * v.x; add[1] += scale * v.y; add[2] += scale * v.z; add[3] += scale * v.w;
            }
            o.x += add[0]; o.y += add[1]; o.z += add[2]; o.w += add[3];
            dst[q] = o;
        }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < T * RG_B * 3; e += RG_BLOCK) {
        const float v = sT[e];
        if (v != 0.f) {
            const int t = e / (RG_B * 3), rem = e % (RG_B * 3), b = rem / 3, d = rem % 3;
            atomicAdd(d_table + ((int64_t)t * RG_B + b) * 7 + d, -v);
            atomicAdd(d_basis_t + b * 7 + d, v);
        }
    }
}

extern "C" int rdg_rigidity_sample(int64_t n, int32_t num_basis, const int32_t* indice, const float* xyz, const float* coeff,
                                   const int32_t* time_ind, const float* basis_t, const float* table, float spatial_lr_scale,
                                   float* points, float* canon, float* coeff_s, void* stream) {
    RDG_CHECK_ARG(n > 0 && indice && xyz && coeff && time_ind && basis_t && table && points && canon && coeff_s, "null argument");
    RDG_CHECK_ARG(num_basis == RG_B, "only num_basis == 16 (the reference's configs) is built");
    RDG_CHECK_ARG((((uintptr_t)coeff | (uintptr_t)coeff_s) & 15) == 0, "coeff buffers must be 16-byte aligned");
    rg_sample_fwd_kernel<<<rdg_div_up(n, RG_BLOCK), RG_BLOCK, 0, (cudaStream_t)stream>>>(
        n, indice, xyz, coeff, time_ind, basis_t, table, spatial_lr_scale, points, canon, coeff_s);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}

extern "C" int rdg_rigidity_sample_bwd(int64_t n, int32_t num_basis, int32_t num_times, const int32_t* indice, const float* coeff,
                                       const int32_t* time_ind, const float* basis_t, const float* table, float spatial_lr_scale,
                                       float grad_scale, const float* d_points, const float* d_canon, const float* d_coeff_s,
                                       float* d_xyz, float* d_coeff, float* d_basis_t, float* d_table, void* stream) {
    RDG_CHECK_ARG(n > 0 && indice && coeff && time_ind && basis_t && table && d_points && d_xyz && d_coeff && d_basis_t && d_table,
                  "null argument");
    RDG_CHECK_ARG(num_basis == RG_B, "only num_basis == 16 (the reference's configs) is built");
    RDG_CHECK_ARG((((uintptr_t)coeff | (uintptr_t)d_coeff | (uintptr_t)d_coeff_s) & 15) == 0, "coeff buffers must be 16-byte aligned");
    const size_t smem = (size_t)num_times * RG_B * 3 * 4;
    RDG_CHECK_ARG(num_times >= 1 && smem <= 160 * 1024, "1 <= num_times <= 853");
    if (smem > 48 * 1024)
        RDG_CUDA(cudaFuncSetAttribute(rg_sample_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t want = (n + RG_BLOCK - 1) / RG_BLOCK;
    const int grid = (int)(want < (int64_t)RDG_SM_COUNT * 2 ? want : (int64_t)RDG_SM_COUNT * 2);
    rg_sample_bwd_kernel<<<grid, RG_BLOCK, smem, (cudaStream_t)stream>>>(n, num_times, indice, coeff, time_ind, basis_t, table,
                                                                          spatial_lr_scale, grad_scale, d_points, d_canon, d_coeff_s,
                                                                          d_xyz, d_coeff, d_basis_t, d_table);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}
