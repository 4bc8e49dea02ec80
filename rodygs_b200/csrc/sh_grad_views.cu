// dL/dSH of ALL camera-time views of a data-parallel step from its rank-1 factors.
// SURVEY.md §8e: the step's views are sharded over the GPUs and the Gaussian-parameter gradients are
// summed.  81 % of that message is dL/dSH [N,16,3], and it is an outer product per view:
//   dL/dSH_i[k][c] = sum_v  Y_k(dir_i,v) * g_i,v[c],     dir_i,v = normalize(x_i(t_v) - campos_v),
// where g_i,v = dL/d(rgb) of Gaussian i in view v after the SH clamp mask (12 bytes).  Every rank holds
// all parameters and all cameras, so it can evaluate Y_k itself: the ranks exchange the 12-byte factors
// (all-gather, written by rdg_preprocess_bwd into RdgSceneGrad.dcolor) instead of all-reducing the
// 192-byte blocks, and this kernel rebuilds the sum over every view.  Same gradient as the sum of the
// per-view dSH that rdg_preprocess_bwd writes on one GPU, up to float summation order.
//
// HBM-bound: reads 12 B (xyz) + 12 B per view [+ 68 B coefficients / birth frame for a dynamic Gaussian],
// writes 12*K B.  One thread per Gaussian, 256-Gaussian chunks of one model; the chunk's 46 KB of dSH
// rows leave through shared memory by one TMA bulk store (coalesced, no LSU store instructions).
#include <stdlib.h>
#include "scene.cuh"
#include "tma.cuh"

#define SH_ROW 45
#define SGV_MAX_VIEWS 16

struct ShAdamSet {
    float* m_dc; float* v_dc;        // [n,3]
    float* m_rest; float* v_rest;    // [n,45]
    float ss_dc, ss_rest;            // lr / (1 - beta1^step)
};

struct ShGradParams {
    RdgScene sc;
    RdgSetGrad st, dy;
    const float* viewmats;   // [V,16] glm storage
    const float* basis_ts;   // [V,K,7] B(t_v) (dynamic + deform only)
    const float* dcolor;     // [V,N,3]
    int n_views;
    int sh_degree;
    float scale;
    int use_tma;
    int tab_smem;            // 1: the translation columns of the whole table are staged in shared memory (num_times <= SGV_TAB_MAX_T)
    uint32_t* sm_queue;      // non-NULL: SM-partitioned mode (see preprocess_bwd.cu): CTAs on SMs >= sm_limit exit, the others share
    int sm_limit;            // a chunk queue, so that a collective on another stream finds free SMs
    // ADAM variant (rdg_sh_adam_views): the rebuilt gradient never leaves the SM - it is consumed by the Adam update of the SH
    // blocks, whose parameters are scene.st / dy.sh_dc, sh_rest themselves
    ShAdamSet ad_st, ad_dy;
    float b1, b2, eps, bc2_sqrt;
    int64_t c_begin, c_end;  // chunk range (one model when only one optimiser steps)
};
#define SGV_TAB_MAX_T 144

// torch.optim.Adam (optim.cu: adam_one) on a contiguous run of floats whose gradient sits in shared memory
__device__ __forceinline__ void sgv_adam_one(float& p, float g, float& m, float& v, float ss, const ShGradParams& a) {
    m = a.b1 * m + (1.f - a.b1) * g;
    v = a.b2 * v + (1.f - a.b2) * g * g;
    const float denom = sqrtf(v) / a.bc2_sqrt + a.eps;
    p -= ss * (m / denom);
}
__device__ __forceinline__ void sgv_adam_run(float* __restrict__ P, float* __restrict__ M, float* __restrict__ V,
                                             const float* __restrict__ g_s, int n_f, float ss, const ShGradParams& a) {
    const int n4 = n_f >> 2;                                  // P, M, V 16-byte aligned (256-Gaussian chunks of 16-byte aligned blocks)
    for (int e = threadIdx.x; e < n4; e += RDG_BLOCK) {
        float4 pp = reinterpret_cast<float4*>(P)[e], mm = __ldcs(reinterpret_cast<const float4*>(M) + e);
        float4 vv = __ldcs(reinterpret_cast<const float4*>(V) + e);
        const float4 g = reinterpret_cast<const float4*>(g_s)[e];
        sgv_adam_one(pp.x, g.x, mm.x, vv.x, ss, a);
        sgv_adam_one(pp.y, g.y, mm.y, vv.y, ss, a);
        sgv_adam_one(pp.z, g.z, mm.z, vv.z, ss, a);
        sgv_adam_one(pp.w, g.w, mm.w, vv.w, ss, a);
        reinterpret_cast<float4*>(P)[e] = pp;
        __stcs(reinterpret_cast<float4*>(M) + e, mm);
        __stcs(reinterpret_cast<float4*>(V) + e, vv);
    }
    const int e = (n4 << 2) + threadIdx.x;                    // ragged tail of the last chunk
    if (e < n_f) sgv_adam_one(P[e], g_s[e], M[e], V[e], ss, a);
}

template <int DEG, bool ADAM>
__global__ void __launch_bounds__(RDG_BLOCK, 2) sh_grad_views_kernel(const ShGradParams p) {
    extern __shared__ __align__(128) float smem[];
    constexpr int K = (DEG + 1) * (DEG + 1);
    const RdgScene& sc = p.sc;
    if (p.sm_queue) {
        unsigned smid;
        asm("mov.u32 %0, %%smid;" : "=r"(smid));
        if ((int)smid >= p.sm_limit) {
            if (threadIdx.x == 0) rdg_queue_release(p.sm_queue, gridDim.x);
            return;
        }
    }
    __shared__ long long q_s[2];
    float* sh_s = smem;                                   // [256][SH_ROW]
    float* coef_s = smem + RDG_BLOCK * SH_ROW;            // [256][17]: the chunk's motion coefficients (coalesced load, padded rows)
    float* tab3_s = coef_s + RDG_BLOCK * 17;              // [T][K][3]: translation columns of the table (tab_smem)
    __shared__ float campos_s[SGV_MAX_VIEWS][3];
    __shared__ float bt3_s[SGV_MAX_VIEWS][RDG_NUM_BASIS_MAX][3];   // B(t_v)[k][0:3]
    __shared__ __align__(16) float dc_s[ADAM ? RDG_BLOCK * 3 : 4];  // ADAM: the chunk's degree-0 gradients
    const bool deform = sc.raw && sc.use_deform && sc.n_dynamic > 0;
    const int nv = p.n_views;
    if ((int)threadIdx.x < nv) {
        // campos = -R^T T of the mathematical V; glm storage: V[r][k] = vm[k*4 + r]
        const float* vm = p.viewmats + threadIdx.x * 16;
#pragma unroll
        for (int j = 0; j < 3; ++j)
            campos_s[threadIdx.x][j] = -(vm[j * 4 + 0] * vm[12 + 0] + vm[j * 4 + 1] * vm[12 + 1] + vm[j * 4 + 2] * vm[12 + 2]);
    }
    if (deform) {
        // all RDG_NUM_BASIS_MAX rows: the per-view sum below runs over every row (c[k] = 0 beyond num_basis), and 0 times a
        // stale NaN / Inf left in shared memory by an earlier kernel is NaN
        for (int e = threadIdx.x; e < nv * RDG_NUM_BASIS_MAX * 3; e += RDG_BLOCK) {
            const int v = e / (RDG_NUM_BASIS_MAX * 3), r = e - v * RDG_NUM_BASIS_MAX * 3, k = r / 3, j = r - k * 3;
            bt3_s[v][k][j] = k < sc.num_basis ? p.basis_ts[((int64_t)v * sc.num_basis + k) * 7 + j] : 0.f;
        }
        // every dynamic Gaussian needs the translation part of its birth-frame row: 48 scattered floats of a 448-byte row per
        // thread from global memory (the L1TEX-bound gather the preprocess kernels got rid of in round 1) - or 19 KB staged once
        if (p.tab_smem)
            for (int e = threadIdx.x; e < sc.num_times * sc.num_basis * 3; e += RDG_BLOCK) {
                const int row = e / 3, j = e - row * 3;
                tab3_s[e] = p.sc.table[(int64_t)row * 7 + j];
            }
    }
    const bool queued = p.sm_queue != nullptr;
    if (queued && threadIdx.x == 0) q_s[0] = p.c_begin + (long long)atomicAdd(p.sm_queue, 1u);
    __syncthreads();

    const int64_t N = sc.n_static + sc.n_dynamic;
    const int64_t cs = (sc.n_static + RDG_BLOCK - 1) / RDG_BLOCK, cd = (sc.n_dynamic + RDG_BLOCK - 1) / RDG_BLOCK;
    bool store_pending = false;
    int q_par = 0;
    for (int64_t chunk = queued ? q_s[0] : p.c_begin + (long long)blockIdx.x; chunk < p.c_end; ) {
        // next chunk: claimed now by thread 0 into the other slot, published by the barrier that precedes the row staging
        q_par ^= 1;
        if (queued && threadIdx.x == 0) q_s[q_par] = p.c_begin + (long long)atomicAdd(p.sm_queue, 1u);
        const bool dyn = chunk >= cs;
        const RdgSet& set = dyn ? sc.dy : sc.st;
        const RdgSetGrad& gs = dyn ? p.dy : p.st;
        const int64_t lbase = (dyn ? chunk - cs : chunk) * RDG_BLOCK;
        const int64_t n_set = dyn ? sc.n_dynamic : sc.n_static;
        const int cnt = (int)min((int64_t)RDG_BLOCK, n_set - lbase);
        const bool valid = (int)threadIdx.x < cnt;
        const int64_t local = lbase + threadIdx.x;
        const int64_t i = (dyn ? sc.n_static : 0) + local;

        const bool def_chunk = deform && dyn;
        if (def_chunk) {
            // coalesced: the chunk's coefficient rows are contiguous in memory; row pitch 17 keeps the per-thread reads conflict-free
            __syncthreads();                               // the previous chunk is done with coef_s
            const float* src = sc.motion_coeff + lbase * sc.num_basis;
            for (int e = threadIdx.x; e < cnt * sc.num_basis; e += RDG_BLOCK) {
                const int gi = e / sc.num_basis, k = e - gi * sc.num_basis;
                coef_s[gi * 17 + k] = __ldg(src + e);
            }
            __syncthreads();
        }
        float g[3 * K];
#pragma unroll
        for (int e = 0; e < 3 * K; ++e) g[e] = 0.f;
        if (valid) {
            const float* px = set.xyz + local * 3;
            float x = __ldg(px), y = __ldg(px + 1), z = __ldg(px + 2);
            float c[RDG_NUM_BASIS_MAX];
            const bool def = deform && dyn;
            if (def) {
                // x(t_v) = x - s sum_k c_k B_k(t_i) + s sum_k c_k B_k(t_v): the birth-frame part once, the view part per view
                const int ti = __ldg(sc.time_ind + local);
                const float* pc = coef_s + threadIdx.x * 17;
                float bx = 0.f, by = 0.f, bz = 0.f;
                if (p.tab_smem) {
                    const float* row = tab3_s + ti * sc.num_basis * 3;
#pragma unroll
                    for (int k = 0; k < RDG_NUM_BASIS_MAX; ++k) {
                        c[k] = k < sc.num_basis ? pc[k] : 0.f;
                        if (k < sc.num_basis) {
                            bx = fmaf(c[k], row[k * 3 + 0], bx);
                            by = fmaf(c[k], row[k * 3 + 1], by);
                            bz = fmaf(c[k], row[k * 3 + 2], bz);
                        }
                    }
                } else {
                    const float* row = sc.table + (int64_t)ti * sc.num_basis * 7;
#pragma unroll
                    for (int k = 0; k < RDG_NUM_BASIS_MAX; ++k) {
                        c[k] = k < sc.num_basis ? pc[k] : 0.f;
                        if (k < sc.num_basis) {
                            bx = fmaf(c[k], __ldg(row + k * 7 + 0), bx);
                            by = fmaf(c[k], __ldg(row + k * 7 + 1), by);
                            bz = fmaf(c[k], __ldg(row + k * 7 + 2), bz);
                        }
                    }
                }
                x -= sc.spatial_lr_scale * bx; y -= sc.spatial_lr_scale * by; z -= sc.spatial_lr_scale * bz;
            }
            // views in groups of four: the twelve factor loads of a group are in flight together (one thread per Gaussian and
            // 16 warps per SM: with one view's loads at a time the kernel sat in long-scoreboard stalls, ncu r02)
            for (int v0 = 0; v0 < nv; v0 += 4) {
                float dcv[4][3];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const bool on = v0 + u < nv;
                    const float* d = p.dcolor + ((int64_t)(on ? v0 + u : v0) * N + i) * 3;
                    dcv[u][0] = on ? __ldg(d) : 0.f;
                    dcv[u][1] = on ? __ldg(d + 1) : 0.f;
                    dcv[u][2] = on ? __ldg(d + 2) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int v = min(v0 + u, nv - 1);
                    const float d0 = dcv[u][0], d1 = dcv[u][1], d2 = dcv[u][2];
                    if (d0 == 0.f && d1 == 0.f && d2 == 0.f) continue;     // not visible in view v (or all channels clamped)
                    float vx = x, vy = y, vz = z;
                    if (def) {
                        float bx = 0.f, by = 0.f, bz = 0.f;
#pragma unroll
                        for (int k = 0; k < RDG_NUM_BASIS_MAX; ++k) {
                            bx = fmaf(c[k], bt3_s[v][k][0], bx);
                            by = fmaf(c[k], bt3_s[v][k][1], by);
                            bz = fmaf(c[k], bt3_s[v][k][2], bz);
                        }
                        vx += sc.spatial_lr_scale * bx; vy += sc.spatial_lr_scale * by; vz += sc.spatial_lr_scale * bz;
                    }
                    float dx = vx - campos_s[v][0], dy = vy - campos_s[v][1], dz = vz - campos_s[v][2];
                    const float inv = rsqrtf(dx * dx + dy * dy + dz * dz);
                    dx *= inv; dy *= inv; dz *= inv;
                    float b[K];
                    rdg_sh_basis<DEG>(dx, dy, dz, b);
#pragma unroll
                    for (int k = 0; k < K; ++k) {
                        g[k * 3 + 0] = fmaf(b[k], d0, g[k * 3 + 0]);
                        g[k * 3 + 1] = fmaf(b[k], d1, g[k * 3 + 1]);
                        g[k * 3 + 2] = fmaf(b[k], d2, g[k * 3 + 2]);
                    }
                }
            }
            if (!ADAM && gs.sh_dc) {
                float* o = gs.sh_dc + local * set.sh_dc_stride;
                o[0] = g[0] * p.scale; o[1] = g[1] * p.scale; o[2] = g[2] * p.scale;
            }
        }
        if (ADAM) {
            // the gradient rows go to shared memory in the parameters' own layout ([cnt][45] and [cnt][3], contiguous in the flat
            // buffer), then the whole CTA streams parameter + two moments through the Adam update with 16-byte accesses
            const ShAdamSet& ad = dyn ? p.ad_dy : p.ad_st;
            __syncthreads();   // the previous chunk's update has read its gradients
            if (valid) {
                float* row = sh_s + threadIdx.x * SH_ROW;
#pragma unroll
                for (int e = 3; e < 3 * K; ++e) row[e - 3] = g[e] * p.scale;
#pragma unroll
                for (int e = 3 * K; e < 48; ++e) row[e - 3] = 0.f;
                dc_s[threadIdx.x * 3 + 0] = g[0] * p.scale;
                dc_s[threadIdx.x * 3 + 1] = g[1] * p.scale;
                dc_s[threadIdx.x * 3 + 2] = g[2] * p.scale;
            }
            __syncthreads();
            sgv_adam_run(const_cast<float*>(set.sh_rest) + lbase * SH_ROW, ad.m_rest + lbase * SH_ROW, ad.v_rest + lbase * SH_ROW,
                         sh_s, cnt * SH_ROW, ad.ss_rest, p);
            sgv_adam_run(const_cast<float*>(set.sh_dc) + lbase * 3, ad.m_dc + lbase * 3, ad.v_dc + lbase * 3, dc_s, cnt * 3, ad.ss_dc, p);
        } else if (gs.sh_rest) {
            const bool tma_out = p.use_tma && set.sh_rest_stride == SH_ROW && (cnt & 3) == 0;
            if (threadIdx.x == 0 && store_pending) { rdg_bulk_store_wait_read(); store_pending = false; }
            __syncthreads();   // the previous chunk's rows have left shared memory
            if (valid) {
                float* row = sh_s + threadIdx.x * SH_ROW;
#pragma unroll
                for (int e = 3; e < 3 * K; ++e) row[e - 3] = g[e] * p.scale;
#pragma unroll
                for (int e = 3 * K; e < 48; ++e) row[e - 3] = 0.f;
            }
            if (tma_out) {
                rdg_fence_proxy_async();
                __syncthreads();
                if (threadIdx.x == 0) {
                    rdg_bulk_store(gs.sh_rest + lbase * SH_ROW, sh_s, (uint32_t)(cnt * SH_ROW * sizeof(float)));
                    store_pending = true;
                }
            } else {
                __syncthreads();
                const int stride = set.sh_rest_stride;
                float* dst = gs.sh_rest + lbase * stride;
                for (int e = threadIdx.x; e < cnt * SH_ROW; e += RDG_BLOCK) {
                    const int gi = e / SH_ROW, k = e - gi * SH_ROW;
                    dst[(int64_t)gi * stride + k] = sh_s[e];
                }
            }
        } else {
            __syncthreads();
        }
        chunk = queued ? q_s[q_par] : chunk + (long long)gridDim.x;
    }
    if (threadIdx.x == 0 && store_pending) rdg_bulk_store_wait_read();
    if (queued && threadIdx.x == 0) rdg_queue_release(p.sm_queue, gridDim.x);
}

// dcolor[i] = acc[i][6..8] with the channels the forward pass clamped at zero masked out: the factors of dL/dSH,
// available as soon as the blend backward is done (so their all-gather overlaps the per-Gaussian backward)
__global__ void __launch_bounds__(RDG_BLOCK) dcolor_from_acc_kernel(int64_t n, const float* __restrict__ acc,
                                                                    const uint8_t* __restrict__ clamped, float* __restrict__ dcolor) {
    for (int64_t i = (int64_t)blockIdx.x * RDG_BLOCK + threadIdx.x; i < n; i += (int64_t)gridDim.x * RDG_BLOCK) {
        const float4 g1 = __ldg(reinterpret_cast<const float4*>(acc + i * 12 + 4));   // dC, dop, dr, dg
        const float gb = __ldg(acc + i * 12 + 8);
        const bool any = g1.z != 0.f || g1.w != 0.f || gb != 0.f;
        const unsigned cl = any ? clamped[i] : 0u;     // only written for visible Gaussians; the others have zero rows
        float* o = dcolor + i * 3;
        o[0] = (cl & 1u) ? 0.f : g1.z;
        o[1] = (cl & 2u) ? 0.f : g1.w;
        o[2] = (cl & 4u) ? 0.f : gb;
    }
}

// The same factors written straight into EVERY rank's gathered buffer: `dcolor_mc` is the NVLink-switch MULTICAST address
// (torch symmetric memory, handle.multicast_ptr) of this rank's block, and multimem.st makes the switch replicate each
// 16-byte store to all GPUs of the group - the all-gather of the data-parallel step fused into the kernel that produces its
// input: one pass, 24 MB of egress per rank instead of seven 24 MB peer copies queued on the copy engines (0.39 ms at 8
// GPUs, profiles/r02_timeline_n8_*.txt).  Four Gaussians per thread = three 16-byte multicast stores.
__device__ __forceinline__ void mc_st_v4(float* addr, float a, float b, float c, float d) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void mc_st_f32(float* addr, float a) {
    asm volatile("multimem.st.relaxed.sys.global.f32 [%0], %1;" ::"l"(addr), "f"(a) : "memory");
}
__global__ void __launch_bounds__(RDG_BLOCK) dcolor_multicast_kernel(int64_t n, const float* __restrict__ acc,
                                                                     const uint8_t* __restrict__ clamped, float* __restrict__ dcolor_mc) {
    const int64_t groups = (n + 3) / 4;
    for (int64_t gq = (int64_t)blockIdx.x * RDG_BLOCK + threadIdx.x; gq < groups; gq += (int64_t)gridDim.x * RDG_BLOCK) {
        float o[12];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t i = gq * 4 + u;
            o[3 * u] = o[3 * u + 1] = o[3 * u + 2] = 0.f;
            if (i < n) {
                const float4 g1 = __ldg(reinterpret_cast<const float4*>(acc + i * 12 + 4));   // dC, dop, dr, dg
                const float gb = __ldg(acc + i * 12 + 8);
                const bool any = g1.z != 0.f || g1.w != 0.f || gb != 0.f;
                const unsigned cl = any ? clamped[i] : 0u;
                o[3 * u] = (cl & 1u) ? 0.f : g1.z;
                o[3 * u + 1] = (cl & 2u) ? 0.f : g1.w;
                o[3 * u + 2] = (cl & 4u) ? 0.f : gb;
            }
        }
        float* dst = dcolor_mc + gq * 12;
        if (gq * 4 + 4 <= n) {
            mc_st_v4(dst, o[0], o[1], o[2], o[3]);
            mc_st_v4(dst + 4, o[4], o[5], o[6], o[7]);
            mc_st_v4(dst + 8, o[8], o[9], o[10], o[11]);
        } else {
            for (int64_t e = 0; e < (n - gq * 4) * 3; ++e) mc_st_f32(dst + e, o[e]);
        }
    }
    __threadfence_system();
}

extern "C" int rdg_dcolor_multicast(int64_t n, const float* acc, const uint8_t* clamped, float* dcolor_mc, void* stream) {
    RDG_CHECK_ARG(acc && clamped && dcolor_mc, "null argument");
    RDG_CHECK_ARG(((uintptr_t)dcolor_mc & 15u) == 0, "the multicast block must be 16-byte aligned");
    if (n <= 0) return RDG_OK;
    const int64_t want = ((n + 3) / 4 + RDG_BLOCK - 1) / RDG_BLOCK;
    const int grid = (int)(want < (int64_t)RDG_SM_COUNT * 8 ? want : (int64_t)RDG_SM_COUNT * 8);
    dcolor_multicast_kernel<<<grid, RDG_BLOCK, 0, (cudaStream_t)stream>>>(n, acc, clamped, dcolor_mc);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}

extern "C" int rdg_dcolor_from_acc(int64_t n, const float* acc, const uint8_t* clamped, float* dcolor, void* stream) {
    RDG_CHECK_ARG(acc && clamped && dcolor, "null argument");
    if (n <= 0) return RDG_OK;
    const int64_t want = (n + RDG_BLOCK - 1) / RDG_BLOCK;
    const int grid = (int)(want < (int64_t)RDG_SM_COUNT * 8 ? want : (int64_t)RDG_SM_COUNT * 8);
    dcolor_from_acc_kernel<<<grid, RDG_BLOCK, 0, (cudaStream_t)stream>>>(n, acc, clamped, dcolor);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}

template <int DEG, bool ADAM>
static int launch_sgv(const ShGradParams& p, int grid, size_t smem, cudaStream_t s) {
    RDG_CUDA(cudaFuncSetAttribute(sh_grad_views_kernel<DEG, ADAM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sh_grad_views_kernel<DEG, ADAM><<<grid, RDG_BLOCK, smem, s>>>(p);
    RDG_CHECK_LAUNCH();
    return RDG_OK;
}

template <bool ADAM>
static int launch_sgv_deg(const ShGradParams& p, int grid, size_t smem, cudaStream_t s) {
    switch (p.sh_degree) {
        case 0: return launch_sgv<0, ADAM>(p, grid, smem, s);
        case 1: return launch_sgv<1, ADAM>(p, grid, smem, s);
        case 2: return launch_sgv<2, ADAM>(p, grid, smem, s);
        default: return launch_sgv<3, ADAM>(p, grid, smem, s);
    }
}

// common argument checks / parameter block of the two entry points
static int sgv_setup(ShGradParams& p, size_t& smem, const RdgScene* scene, int32_t sh_degree, int32_t n_views,
                     const float* viewmatrices, const float* basis_ts, const float* dcolor, float scale, const char* who) {
    (void)who;
    RDG_CHECK_ARG(scene && viewmatrices && dcolor, "null argument");
    RDG_CHECK_ARG(n_views > 0 && n_views <= SGV_MAX_VIEWS, "n_views must be 1..16");
    RDG_CHECK_ARG(sh_degree >= 0 && sh_degree <= 3, "sh_degree must be 0..3");
    const bool deform = scene->raw && scene->use_deform && scene->n_dynamic > 0;
    if (deform) {
        RDG_CHECK_ARG(scene->num_basis > 0 && scene->num_basis <= RDG_NUM_BASIS_MAX, "num_basis out of range");
        RDG_CHECK_ARG(scene->motion_coeff && scene->time_ind && scene->table && basis_ts, "null deformation input");
    }
    RDG_CHECK_ARG((scene->n_static == 0 || scene->st.xyz) && (scene->n_dynamic == 0 || scene->dy.xyz), "null means");
    p.sc = *scene;
    p.st = RdgSetGrad{}; p.dy = RdgSetGrad{};
    p.ad_st = ShAdamSet{}; p.ad_dy = ShAdamSet{};
    p.b1 = p.b2 = p.eps = p.bc2_sqrt = 0.f;
    p.viewmats = viewmatrices; p.basis_ts = basis_ts; p.dcolor = dcolor;
    p.n_views = n_views; p.sh_degree = sh_degree; p.scale = scale;
    p.use_tma = 0;
    p.tab_smem = (deform && scene->num_times <= SGV_TAB_MAX_T) ? 1 : 0;
    p.sm_queue = nullptr;
    p.sm_limit = 0;
    p.c_begin = 0;
    p.c_end = (scene->n_static + RDG_BLOCK - 1) / RDG_BLOCK + (scene->n_dynamic + RDG_BLOCK - 1) / RDG_BLOCK;
    smem = ((size_t)RDG_BLOCK * SH_ROW + (size_t)RDG_BLOCK * 17 +
            (p.tab_smem ? (size_t)scene->num_times * scene->num_basis * 3 : 0)) * sizeof(float);
    return RDG_OK;
}

extern "C" int rdg_sh_grad_views(const RdgScene* scene, int32_t sh_degree, int32_t n_views, const float* viewmatrices,
                                 const float* basis_ts, const float* dcolor, float scale, const RdgSetGrad* grad_static,
                                 const RdgSetGrad* grad_dynamic, uint32_t* sm_queue, void* stream) {
    RDG_CHECK_ARG(grad_static && grad_dynamic, "null argument");
    ShGradParams p;
    size_t smem;
    const int rc0 = sgv_setup(p, smem, scene, sh_degree, n_views, viewmatrices, basis_ts, dcolor, scale, "rdg_sh_grad_views");
    if (rc0) return rc0;
    if (scene->n_static + scene->n_dynamic == 0) return RDG_OK;
    p.st = *grad_static; p.dy = *grad_dynamic;
    p.use_tma = ((((uintptr_t)grad_static->sh_rest | (uintptr_t)grad_dynamic->sh_rest) & 15u) == 0) ? 1 : 0;
    const int64_t chunks = p.c_end - p.c_begin;
    // persistent grid, two CTAs per SM.  "sm_reserve" leaves SMs to a collective that runs at the same time - these CTAs
    // take the whole register file of the SMs they sit on.
    int sms = RDG_SM_COUNT - rdg_tunable(RDG_TUN_SM_RESERVE);
    if (sms < 8) sms = 8;
    const int64_t cap = (int64_t)sms * 2;
    int grid = (int)(chunks < cap ? chunks : cap);
    cudaStream_t s = (cudaStream_t)stream;
    if (sm_queue && sms < RDG_SM_COUNT && chunks > cap) {
        p.sm_queue = sm_queue;             // zero on entry, left zero by the kernel (rdg_queue_release)
        p.sm_limit = sms;
        grid = RDG_SM_COUNT * 2;
    }
    const int rc = launch_sgv_deg<false>(p, grid, smem, s);
    if (rc) return rc;
    rdg_count_launches(1);
    return RDG_OK;
}

// The same sum over views, consumed where it is produced: Adam over the SH blocks (f_dc / f_rest groups of one or both
// models) with the gradient rebuilt per 256-Gaussian chunk in shared memory.  The 192-byte dL/dSH blocks - 81 % of the
// gradient buffer - are never written to or read back from HBM.
extern "C" int rdg_sh_adam_views(const RdgScene* scene, int32_t sh_degree, int32_t n_views, const float* viewmatrices,
                                 const float* basis_ts, const float* dcolor, float scale, const RdgShAdam* adam_static,
                                 const RdgShAdam* adam_dynamic, float beta1, float beta2, float eps, void* stream) {
    ShGradParams p;
    size_t smem;
    const int rc0 = sgv_setup(p, smem, scene, sh_degree, n_views, viewmatrices, basis_ts, dcolor, scale, "rdg_sh_adam_views");
    if (rc0) return rc0;
    const bool on_st = adam_static && adam_static->step > 0 && scene->n_static > 0;
    const bool on_dy = adam_dynamic && adam_dynamic->step > 0 && scene->n_dynamic > 0;
    if (!on_st && !on_dy) return RDG_OK;
    const int64_t cs = (scene->n_static + RDG_BLOCK - 1) / RDG_BLOCK;
    auto fill = [&](ShAdamSet& o, const RdgShAdam* a, const RdgSet& set) -> int {
        RDG_CHECK_ARG(a->exp_avg_dc && a->exp_avg_sq_dc && a->exp_avg_rest && a->exp_avg_sq_rest, "null moment buffer");
        RDG_CHECK_ARG(set.sh_dc && set.sh_rest && set.sh_dc_stride == 3 && set.sh_rest_stride == SH_ROW,
                      "the SH blocks must be the contiguous [n,3] / [n,45] parameter tensors");
        RDG_CHECK_ARG((((uintptr_t)set.sh_dc | (uintptr_t)set.sh_rest | (uintptr_t)a->exp_avg_dc | (uintptr_t)a->exp_avg_sq_dc |
                        (uintptr_t)a->exp_avg_rest | (uintptr_t)a->exp_avg_sq_rest) & 15u) == 0, "buffers must be 16-byte aligned");
        const float bc1 = 1.0f - (float)pow((double)beta1, (double)a->step);
        o.m_dc = a->exp_avg_dc; o.v_dc = a->exp_avg_sq_dc; o.m_rest = a->exp_avg_rest; o.v_rest = a->exp_avg_sq_rest;
        o.ss_dc = a->lr_dc / bc1;
        o.ss_rest = a->lr_rest / bc1;
        return RDG_OK;
    };
    int step = 0;
    if (on_st) { const int rc = fill(p.ad_st, adam_static, scene->st); if (rc) return rc; step = adam_static->step; }
    if (on_dy) { const int rc = fill(p.ad_dy, adam_dynamic, scene->dy); if (rc) return rc; step = adam_dynamic->step; }
    RDG_CHECK_ARG(!(on_st && on_dy) || adam_static->step == adam_dynamic->step,
                  "both models in one launch must be at the same step (bias correction); call once per model otherwise");
    p.b1 = beta1; p.b2 = beta2; p.eps = eps;
    p.bc2_sqrt = sqrtf(1.0f - (float)pow((double)beta2, (double)step));
    if (!on_st) p.c_begin = cs;
    if (!on_dy) p.c_end = cs;
    const int64_t chunks = p.c_end - p.c_begin;
    const int64_t cap = (int64_t)RDG_SM_COUNT * 2;
    const int grid = (int)(chunks < cap ? chunks : cap);
    const int rc = launch_sgv_deg<true>(p, grid, smem, (cudaStream_t)stream);
    if (rc) return rc;
    rdg_count_launches(1);
    return RDG_OK;
}
