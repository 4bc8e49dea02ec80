// Point tracking through the learned motion: where a pixel of a source render goes at a target time, seen from a target
// camera (INTEGRATION.md §10).
//
//   rdg_track_attrs   puts each visible Gaussian's target-time centre mu_k(t_m) into its record's colour slots (p1.z, p1.w,
//                     p2.x), so that rdg_blend_fwd over the source view's bins - the path colors_precomp takes, unclamped -
//                     blends S_m(p) = sum_k w_k(p) mu_k(t_m) with the source render's exact weights.
//   rdg_track_project normalises S_m by the source alpha and projects the tracked point into each target camera, densely
//                     (every pixel) or at sparse query points (bilinear between pixel centres).
//
// THIS TRANSLATION UNIT IS COMPILED WITH -fmad=false, like preprocess_fwd.cu: the deformation rounds every operation the
// way the preprocess does (its explicit fmaf chain included), so mu_k(t_s) here has the bits of the preprocess's deformed
// mean, and the projection has rdg_project's operation order.
#include "scene.cuh"

// largest T whose table rows are staged in shared memory (the limit of rdg_preprocess_fwd_views, so that T = 137 / 138
// covers both table paths of both kernels); above it each dynamic Gaussian gathers its row from global memory
#define RDG_TRACK_TABLE_MAX 137

struct TrackAttrsParams {
    RdgScene sc;
    const float* basis_t;   // B(t_m) [num_basis, 7]
    RdgGeom geom;
    float* positions;       // optional [N, 3]
    int diff_smem;          // B(t_m) - table rows staged in shared memory (rdg_stage_diff)
};

// Roofline: HBM.  Per Gaussian read 4 (radius) + 12 (xyz) [+ 68 dynamic: coefficients + birth index, only when it is
// visible or positions is set], write 12 when visible (+ 12 to positions).
__global__ void __launch_bounds__(RDG_BLOCK) track_attrs_kernel(const TrackAttrsParams p) {
    extern __shared__ __align__(16) float diff_s[];   // [T][RDG_DIFF_STRIDE] when p.diff_smem
    const RdgScene& sc = p.sc;
    const bool deform = sc.raw && sc.use_deform && sc.n_dynamic > 0;
    if (deform && p.diff_smem) {
        rdg_stage_diff(sc, p.basis_t, diff_s, RDG_BLOCK);
        __syncthreads();
    }
    const int64_t cs = (sc.n_static + RDG_BLOCK - 1) / RDG_BLOCK, cd = (sc.n_dynamic + RDG_BLOCK - 1) / RDG_BLOCK;
    for (int64_t chunk = blockIdx.x; chunk < cs + cd; chunk += gridDim.x) {
        const bool dyn = chunk >= cs;
        const int64_t local = (dyn ? chunk - cs : chunk) * RDG_BLOCK + threadIdx.x;
        if (local >= (dyn ? sc.n_dynamic : sc.n_static)) continue;
        const int64_t i = (dyn ? sc.n_static : 0) + local;
        const bool vis = __ldg(p.geom.radii + i) > 0;
        if (!vis && !p.positions) continue;
        const float* px = (dyn ? sc.dy.xyz : sc.st.xyz) + local * 3;
        RdgAct a;
        a.x = __ldg(px); a.y = __ldg(px + 1); a.z = __ldg(px + 2);
        a.q[0] = a.q[1] = a.q[2] = a.q[3] = 0.f;
        if (deform && dyn) {
            // the coefficient load and delta of rdg_fetch<RAW = true>, at B(t_m)
            float c[RDG_NUM_BASIS_MAX];
            const float* pc = sc.motion_coeff + local * sc.num_basis;
            if (sc.num_basis == RDG_NUM_BASIS_MAX) {
                const float4* pc4 = reinterpret_cast<const float4*>(pc);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 v = __ldg(pc4 + q);
                    c[4 * q] = v.x; c[4 * q + 1] = v.y; c[4 * q + 2] = v.z; c[4 * q + 3] = v.w;
                }
            } else {
#pragma unroll
                for (int k = 0; k < RDG_NUM_BASIS_MAX; ++k) c[k] = k < sc.num_basis ? __ldg(pc + k) : 0.f;
            }
            float d[7];
            rdg_deform_delta(sc, p.basis_t, __ldg(sc.time_ind + local), c, d, p.diff_smem ? diff_s : nullptr);
            rdg_apply_deform(sc, d, a);
        }
        if (vis) {
            reinterpret_cast<float2*>(p.geom.p1)[2 * i + 1] = make_float2(a.x, a.y);   // p1.z, p1.w
            p.geom.p2[2 * i] = a.z;                                                      // p2.x
        }
        if (p.positions) {
            float* o = p.positions + i * 3;
            o[0] = a.x; o[1] = a.y; o[2] = a.z;
        }
    }
}

extern "C" int rdg_track_attrs(const RdgScene* scene, const float* basis_t_target, const RdgGeom* geom, float* positions_out,
                               void* stream) {
    RDG_CHECK_ARG(scene && geom, "null argument");
    RDG_CHECK_ARG(scene->basis_t == nullptr, "scene->basis_t must be NULL: B(t) of the target comes from basis_t_target");
    RDG_CHECK_ARG(scene->n_static >= 0 && scene->n_dynamic >= 0, "negative count");
    const int64_t N = scene->n_static + scene->n_dynamic;
    if (N == 0) return RDG_OK;
    RDG_CHECK_ARG(geom->radii && geom->p1 && geom->p2, "null geometry buffer");
    RDG_CHECK_ARG(scene->n_static == 0 || scene->st.xyz, "null static parameter");
    RDG_CHECK_ARG(scene->n_dynamic == 0 || scene->dy.xyz, "null dynamic parameter");
    const bool deform = scene->raw && scene->use_deform && scene->n_dynamic > 0;
    if (deform) {
        RDG_CHECK_ARG(scene->num_basis > 0 && scene->num_basis <= RDG_NUM_BASIS_MAX, "num_basis out of range");
        RDG_CHECK_ARG(scene->motion_coeff && scene->time_ind && basis_t_target && scene->table && scene->num_times > 0,
                      "null deformation input");
    }
    TrackAttrsParams p;
    p.sc = *scene;
    p.basis_t = basis_t_target;
    p.geom = *geom;
    p.positions = positions_out;
    p.diff_smem = 0;
    size_t smem = 0;
    if (deform && scene->num_basis == RDG_NUM_BASIS_MAX && scene->num_times <= RDG_TRACK_TABLE_MAX &&
        (((uintptr_t)basis_t_target | (uintptr_t)scene->table) & 15u) == 0) {
        p.diff_smem = 1;
        smem = (size_t)scene->num_times * RDG_DIFF_STRIDE * sizeof(float);
    }
    // persistent grid, so that each CTA stages the difference table once: 3 CTAs per SM fit beside the largest staged table
    // (64 KB each), 4 without one (registers: `-Xptxas -v` shows 55)
    const int64_t chunks = (scene->n_static + RDG_BLOCK - 1) / RDG_BLOCK + (scene->n_dynamic + RDG_BLOCK - 1) / RDG_BLOCK;
    const int64_t per_sm = p.diff_smem ? 3 : 4;
    const int grid = (int)(chunks < (int64_t)RDG_SM_COUNT * per_sm ? chunks : (int64_t)RDG_SM_COUNT * per_sm);
    RDG_CUDA(cudaFuncSetAttribute(track_attrs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    track_attrs_kernel<<<grid, RDG_BLOCK, smem, (cudaStream_t)stream>>>(p);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}

// ---- normalise + project ----

struct TrackProjectParams {
    const float* S;          // [M, 3, H, W]
    const float* A;          // [H, W]
    const float* viewmats;   // [M, 16] glm storage
    const float* projmats;   // [M, 16] glm storage
    const float* points;     // [P, 2] or NULL (dense)
    float* xy;               // dense [M, 2, H, W], sparse [M, P, 2]
    float* depth;            // dense [M, 1, H, W], sparse [M, P]
    float* alpha;            // sparse only, optional: [P] the sampled A
    int H, W;
    int64_t count;           // H * W (dense) or P (sparse)
};

// X = s / a, v = V X, c = P v, ndc = c.xy / (c.w + 1e-7) in rdg_project's operation order; NaN everywhere where a == 0
__device__ __forceinline__ void rdg_track_point(const float* vm, const float* pm, float sx, float sy, float sz, float a,
                                                float W, float H, float& px, float& py, float& depth) {
    if (a == 0.0f) {
        px = py = depth = __int_as_float(0x7fffffff);
        return;
    }
    const float x = sx / a, y = sy / a, z = sz / a;
    // glm storage: element (r, k) of the mathematical matrix sits at [k * 4 + r]
    const float tx = __ldg(vm + 0) * x + __ldg(vm + 4) * y + __ldg(vm + 8) * z + __ldg(vm + 12);
    const float ty = __ldg(vm + 1) * x + __ldg(vm + 5) * y + __ldg(vm + 9) * z + __ldg(vm + 13);
    const float tz = __ldg(vm + 2) * x + __ldg(vm + 6) * y + __ldg(vm + 10) * z + __ldg(vm + 14);
    const float hx = __ldg(pm + 0) * tx + __ldg(pm + 4) * ty + __ldg(pm + 8) * tz + __ldg(pm + 12);
    const float hy = __ldg(pm + 1) * tx + __ldg(pm + 5) * ty + __ldg(pm + 9) * tz + __ldg(pm + 13);
    const float hw = __ldg(pm + 3) * tx + __ldg(pm + 7) * ty + __ldg(pm + 11) * tz + __ldg(pm + 15);
    const float pw = 1.0f / (hw + 0.0000001f);
    const float ndcx = hx * pw, ndcy = hy * pw;
    px = ((ndcx + 1.0f) * W - 1.0f) * 0.5f;
    py = ((ndcy + 1.0f) * H - 1.0f) * 0.5f;
    depth = tz;
}

// a + f (b - a): f = 0 returns a's bits
__device__ __forceinline__ float rdg_lerp(float a, float b, float f) { return a + f * (b - a); }

// one thread per (target, pixel) or (target, point); blockIdx.y = target.  No atomics: every output has one writer.
template <bool SPARSE>
__global__ void __launch_bounds__(RDG_BLOCK) track_project_kernel(const TrackProjectParams p) {
    const int64_t e = (int64_t)blockIdx.x * RDG_BLOCK + threadIdx.x;
    if (e >= p.count) return;
    const int m = blockIdx.y;
    const int64_t HW = (int64_t)p.H * p.W;
    const float* S = p.S + (int64_t)m * 3 * HW;
    float s0, s1, s2, a;
    if (!SPARSE) {
        s0 = S[e]; s1 = S[HW + e]; s2 = S[2 * HW + e];
        a = p.A[e];
    } else {
        // bilinear between pixel centres (pixel (x, y) is centred at integer x, y), clamped to the image; a NaN coordinate
        // fails both comparisons and stays NaN, so its outputs are NaN
        float x = __ldg(p.points + 2 * e), y = __ldg(p.points + 2 * e + 1);
        const float xmax = (float)(p.W - 1), ymax = (float)(p.H - 1);
        x = x < 0.0f ? 0.0f : (x > xmax ? xmax : x);
        y = y < 0.0f ? 0.0f : (y > ymax ? ymax : y);
        const float fx0 = floorf(x), fy0 = floorf(y);
        const int x0 = min(max((int)fx0, 0), p.W - 1), y0 = min(max((int)fy0, 0), p.H - 1);
        const int x1 = min(x0 + 1, p.W - 1), y1 = min(y0 + 1, p.H - 1);
        const float fx = x - fx0, fy = y - fy0;
        const int64_t i00 = (int64_t)y0 * p.W + x0, i01 = (int64_t)y0 * p.W + x1;
        const int64_t i10 = (int64_t)y1 * p.W + x0, i11 = (int64_t)y1 * p.W + x1;
        float v[4];
        const float* src[4] = {S, S + HW, S + 2 * HW, p.A};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const float* q = src[c];
            v[c] = rdg_lerp(rdg_lerp(q[i00], q[i01], fx), rdg_lerp(q[i10], q[i11], fx), fy);
        }
        s0 = v[0]; s1 = v[1]; s2 = v[2]; a = v[3];
        if (m == 0 && p.alpha) p.alpha[e] = a;
    }
    float px, py, d;
    rdg_track_point(p.viewmats + m * 16, p.projmats + m * 16, s0, s1, s2, a, (float)p.W, (float)p.H, px, py, d);
    if (!SPARSE) {
        float* xy = p.xy + (int64_t)m * 2 * HW;
        xy[e] = px;
        xy[HW + e] = py;
        p.depth[(int64_t)m * HW + e] = d;
    } else {
        reinterpret_cast<float2*>(p.xy)[(int64_t)m * p.count + e] = make_float2(px, py);
        p.depth[(int64_t)m * p.count + e] = d;
    }
}

extern "C" int rdg_track_project(const float* S, const float* A, int32_t M, int32_t height, int32_t width,
                                 const float* viewmats, const float* projmats, const float* points, int64_t P, float* xy_out,
                                 float* depth_out, float* alpha_out, void* stream) {
    RDG_CHECK_ARG(S && A && viewmats && projmats && xy_out && depth_out, "null argument");
    RDG_CHECK_ARG(height > 0 && width > 0, "empty image");
    RDG_CHECK_ARG(M >= 1 && M <= 65535, "M must be 1..65535");
    RDG_CHECK_ARG(P >= 0, "negative point count");
    TrackProjectParams p;
    p.S = S; p.A = A; p.viewmats = viewmats; p.projmats = projmats; p.points = points;
    p.xy = xy_out; p.depth = depth_out; p.alpha = alpha_out;
    p.H = height; p.W = width;
    p.count = points ? P : (int64_t)height * width;
    if (p.count == 0) return RDG_OK;
    const dim3 grid((unsigned)((p.count + RDG_BLOCK - 1) / RDG_BLOCK), (unsigned)M);
    if (points) track_project_kernel<true><<<grid, RDG_BLOCK, 0, (cudaStream_t)stream>>>(p);
    else track_project_kernel<false><<<grid, RDG_BLOCK, 0, (cudaStream_t)stream>>>(p);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}
