// Export of a scene at one time t as the records of 3D Gaussian Splatting's PLY file (INTEGRATION.md §11).
//
//   rdg_export_3dgs writes one 62-float record per Gaussian, static rows first, in the property order of 3DGS's
//                   construct_list_of_attributes: x y z nx ny nz f_dc_0..2 f_rest_0..44 opacity scale_0..2 rot_0..3.
//
// A dynamic Gaussian's quaternion q' = normalize(q) + dq(t) is not re-normalised, and rdg_project builds R(q') with the
// unit-quaternion formula, so R(q') is not a rotation when |q'| != 1.  A viewer normalises whatever quaternion it reads, so
// q' cannot be written as it is: the record holds the covariance the rasterizer draws, Sigma = R(q') S^2 R(q')^T, factored
// again (float64 Jacobi) into a unit quaternion and log-scales.
//
// THIS TRANSLATION UNIT IS COMPILED WITH -fmad=false, like preprocess_fwd.cu and track.cu: the deformation rounds every
// operation the way the preprocess does, so the deformed mean has the bits of the preprocess's.
#include <float.h>
#include "scene.cuh"

// largest T whose B(t) - table rows are staged in shared memory (rdg_stage_diff), as in track.cu; above it each dynamic
// Gaussian gathers its table row from global memory
#define RDG_EXPORT_TABLE_MAX 137
// per Gaussian, staged for the coalesced copy-out: x y z, opacity, scale_0..2, rot_0..3 (odd stride: no bank conflicts)
#define RDG_EXPORT_STAGE 11

struct ExportParams {
    RdgScene sc;
    float* records;    // [N, RDG_3DGS_RECORD_FLOATS]
    int rest_coeffs;   // (sh_degree + 1)^2 - 1 higher-order coefficients are copied, the others written as 0
    int diff_smem;     // B(t) - table rows staged in shared memory (rdg_stage_diff)
};

// One Jacobi rotation of the symmetric A in the (P, Q) plane that zeroes A[P][Q] (Numerical Recipes' jacobi, float64);
// V accumulates the rotations, so its columns are the eigenvectors and det V = +1.
template <int P, int Q>
__device__ __forceinline__ void rdg_jacobi_rotate(double (&A)[3][3], double (&V)[3][3]) {
    constexpr int K = 3 - P - Q;
    const double apq = A[P][Q];
    if (apq == 0.0) return;
    const double theta = (A[Q][Q] - A[P][P]) / (2.0 * apq);
    const double at = fabs(theta);
    double t = at > 1e150 ? 0.5 / at : 1.0 / (at + sqrt(at * at + 1.0));   // the smaller root of t^2 + 2 theta t - 1
    if (theta < 0.0) t = -t;
    const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
    A[P][P] -= t * apq;
    A[Q][Q] += t * apq;
    A[P][Q] = A[Q][P] = 0.0;
    const double akp = A[K][P], akq = A[K][Q];
    A[K][P] = A[P][K] = c * akp - s * akq;
    A[K][Q] = A[Q][K] = s * akp + c * akq;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double vp = V[k][P], vq = V[k][Q];
        V[k][P] = c * vp - s * vq;
        V[k][Q] = s * vp + c * vq;
    }
}

// Sigma = M M^T, M = R(q) diag(s) with rdg_project's R (the unit-quaternion formula, q as it is), in float64; then
// Sigma = U diag(lambda) U^T, rot = the unit quaternion of U with rot[0] >= 0 and scale_j = 0.5 log(max(lambda_j, FLT_MIN)).
// Deterministic: cyclic sweeps until the off-diagonal part is below 1e-16 of the diagonal (at most 12 sweeps).
__device__ __forceinline__ void rdg_export_factor(const float* q, const float* s, float* rot, float* scale) {
    const double qr = q[0], qx = q[1], qy = q[2], qz = q[3];
    const double R[3][3] = {{1.0 - 2.0 * (qy * qy + qz * qz), 2.0 * (qx * qy - qr * qz), 2.0 * (qx * qz + qr * qy)},
                            {2.0 * (qx * qy + qr * qz), 1.0 - 2.0 * (qx * qx + qz * qz), 2.0 * (qy * qz - qr * qx)},
                            {2.0 * (qx * qz - qr * qy), 2.0 * (qy * qz + qr * qx), 1.0 - 2.0 * (qx * qx + qy * qy)}};
    const double sd[3] = {s[0], s[1], s[2]};
    double A[3][3], V[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            A[i][j] = (R[i][0] * sd[0]) * (R[j][0] * sd[0]) + (R[i][1] * sd[1]) * (R[j][1] * sd[1]) +
                      (R[i][2] * sd[2]) * (R[j][2] * sd[2]);
            V[i][j] = i == j ? 1.0 : 0.0;
        }
#pragma unroll 1
    for (int sweep = 0; sweep < 12; ++sweep) {
        const double off = A[0][1] * A[0][1] + A[0][2] * A[0][2] + A[1][2] * A[1][2];
        const double diag = A[0][0] * A[0][0] + A[1][1] * A[1][1] + A[2][2] * A[2][2];
        if (off <= 1e-32 * diag) break;   // also ends a zero Sigma at once
        rdg_jacobi_rotate<0, 1>(A, V);
        rdg_jacobi_rotate<0, 2>(A, V);
        rdg_jacobi_rotate<1, 2>(A, V);
    }
    // quaternion of the rotation U = V (Shepperd: divide by the largest of 4w^2, 4x^2, 4y^2, 4z^2)
    const double tr = V[0][0] + V[1][1] + V[2][2];
    double w, x, y, z;
    if (tr > 0.0) {
        const double f = 2.0 * sqrt(tr + 1.0);
        w = 0.25 * f; x = (V[2][1] - V[1][2]) / f; y = (V[0][2] - V[2][0]) / f; z = (V[1][0] - V[0][1]) / f;
    } else if (V[0][0] > V[1][1] && V[0][0] > V[2][2]) {
        const double f = 2.0 * sqrt(1.0 + V[0][0] - V[1][1] - V[2][2]);
        w = (V[2][1] - V[1][2]) / f; x = 0.25 * f; y = (V[0][1] + V[1][0]) / f; z = (V[0][2] + V[2][0]) / f;
    } else if (V[1][1] > V[2][2]) {
        const double f = 2.0 * sqrt(1.0 + V[1][1] - V[0][0] - V[2][2]);
        w = (V[0][2] - V[2][0]) / f; x = (V[0][1] + V[1][0]) / f; y = 0.25 * f; z = (V[1][2] + V[2][1]) / f;
    } else {
        const double f = 2.0 * sqrt(1.0 + V[2][2] - V[0][0] - V[1][1]);
        w = (V[1][0] - V[0][1]) / f; x = (V[0][2] + V[2][0]) / f; y = (V[1][2] + V[2][1]) / f; z = 0.25 * f;
    }
    const double inv = (w < 0.0 ? -1.0 : 1.0) / sqrt(w * w + x * x + y * y + z * z);
    rot[0] = (float)(w * inv); rot[1] = (float)(x * inv); rot[2] = (float)(y * inv); rot[3] = (float)(z * inv);
#pragma unroll
    for (int j = 0; j < 3; ++j) scale[j] = (float)(0.5 * log(fmax(A[j][j], (double)FLT_MIN)));
}

// Field f (0..61) of the record of Gaussian g of the chunk: geometry from the stage, SH from the parameters (transposed to
// channel-major, zero above the degree).
__device__ __forceinline__ float rdg_export_field(const ExportParams& p, const RdgSet& set, const float* stage, int64_t row,
                                                  int g, int f) {
    if (f < 3) return stage[g * RDG_EXPORT_STAGE + f];                               // x y z
    if (f < 6) return 0.0f;                                                           // nx ny nz
    if (f < 9) return __ldg(set.sh_dc + row * set.sh_dc_stride + (f - 6));           // f_dc_c
    if (f < 54) {                                                                     // f_rest_{15 c + k - 1}
        const int j = f - 9, c = j / 15, k1 = j - 15 * c;
        return k1 < p.rest_coeffs ? __ldg(set.sh_rest + row * set.sh_rest_stride + 3 * k1 + c) : 0.0f;
    }
    return stage[g * RDG_EXPORT_STAGE + (f - 51)];                                   // opacity scale_0..2 rot_0..3
}

// Roofline: HBM.  Per Gaussian read 44 (xyz, log-scale, rotation, opacity) + 4 (sh_rest_coeffs + 1) x 3 of SH [+ 68
// dynamic: coefficients + birth index], write 248.  The float64 factorisation of the dynamic rows is the compute part.
__global__ void __launch_bounds__(RDG_BLOCK, 2) export_3dgs_kernel(const ExportParams p) {
    extern __shared__ __align__(16) float diff_s[];   // [T][RDG_DIFF_STRIDE] when p.diff_smem
    __shared__ float stage[RDG_BLOCK * RDG_EXPORT_STAGE];
    const RdgScene& sc = p.sc;
    if (p.diff_smem) {
        rdg_stage_diff(sc, sc.basis_t, diff_s, RDG_BLOCK);
        __syncthreads();
    }
    const int64_t cs = (sc.n_static + RDG_BLOCK - 1) / RDG_BLOCK, cd = (sc.n_dynamic + RDG_BLOCK - 1) / RDG_BLOCK;
    for (int64_t chunk = blockIdx.x; chunk < cs + cd; chunk += gridDim.x) {
        const bool dyn = chunk >= cs;
        const RdgSet& set = dyn ? sc.dy : sc.st;
        const int64_t lbase = (dyn ? chunk - cs : chunk) * RDG_BLOCK;
        const int cnt = (int)min((int64_t)RDG_BLOCK, (dyn ? sc.n_dynamic : sc.n_static) - lbase);
        if ((int)threadIdx.x < cnt) {
            const int64_t local = lbase + threadIdx.x;
            float* st = stage + threadIdx.x * RDG_EXPORT_STAGE;
            st[3] = __ldg(set.opacity + local);                                        // the raw logit, both sets
            if (!dyn) {                                                                 // the raw parameters, bit for bit
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    st[j] = __ldg(set.xyz + local * 3 + j);
                    st[4 + j] = __ldg(set.scaling + local * 3 + j);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) st[7 + j] = __ldg(set.rotation + local * 4 + j);
            } else {
                // rdg_fetch<RAW = true, DEFORM = true>'s loads, activations and deformation, written out as in track.cu
                // (rdg_fetch itself keeps a 144-byte stack frame here)
                RdgAct a;
                a.x = __ldg(set.xyz + local * 3); a.y = __ldg(set.xyz + local * 3 + 1); a.z = __ldg(set.xyz + local * 3 + 2);
#pragma unroll
                for (int j = 0; j < 3; ++j) a.s[j] = expf(__ldg(set.scaling + local * 3 + j));
                const float4 q4 = __ldg(reinterpret_cast<const float4*>(set.rotation) + local);
                const float qinv = 1.0f / fmaxf(sqrtf(q4.x * q4.x + q4.y * q4.y + q4.z * q4.z + q4.w * q4.w), 1e-12f);
                a.q[0] = q4.x * qinv; a.q[1] = q4.y * qinv; a.q[2] = q4.z * qinv; a.q[3] = q4.w * qinv;
                if (sc.use_deform) {
                    // the coefficients are read where they are, not through a register array: the delta's general loop
                    // (num_basis < 16) indexes them at run time, which would put such an array on a stack frame.  The
                    // same floats go into the same operations.
                    float d[7];
                    rdg_deform_delta(sc, sc.basis_t, __ldg(sc.time_ind + local), sc.motion_coeff + local * sc.num_basis, d,
                                     p.diff_smem ? diff_s : nullptr);
                    rdg_apply_deform(sc, d, a);
                }
                st[0] = a.x; st[1] = a.y; st[2] = a.z;
                rdg_export_factor(a.q, a.s, st + 7, st + 4);
            }
        }
        __syncthreads();
        // copy-out: the chunk's records are one contiguous range; consecutive threads write consecutive float pairs
        float2* out = reinterpret_cast<float2*>(p.records + ((dyn ? sc.n_static : 0) + lbase) * RDG_3DGS_RECORD_FLOATS);
        const int half = RDG_3DGS_RECORD_FLOATS / 2;
        for (int e = threadIdx.x; e < cnt * half; e += RDG_BLOCK) {
            const int g = e / half, f = 2 * (e - g * half);
            out[e] = make_float2(rdg_export_field(p, set, stage, lbase + g, g, f),
                                 rdg_export_field(p, set, stage, lbase + g, g, f + 1));
        }
        __syncthreads();
    }
}

extern "C" int rdg_export_3dgs(const RdgScene* scene, int32_t sh_degree, float* records, void* stream) {
    RDG_CHECK_ARG(scene, "null argument");
    RDG_CHECK_ARG(scene->n_static >= 0 && scene->n_dynamic >= 0, "negative count");
    RDG_CHECK_ARG(scene->raw == 1, "raw must be 1: the record is defined from the raw parameters");
    RDG_CHECK_ARG(scene->colors_precomp == nullptr, "colors_precomp must be NULL: the record holds SH coefficients");
    RDG_CHECK_ARG(sh_degree >= 0 && sh_degree <= 3, "sh_degree must be 0..3");
    const int64_t N = scene->n_static + scene->n_dynamic;
    if (N == 0) return RDG_OK;
    RDG_CHECK_ARG(records, "null argument");
    RDG_CHECK_ARG(((uintptr_t)records & 7u) == 0, "records must be 8-byte aligned");
    const RdgSet* sets[2] = {&scene->st, &scene->dy};
    const int64_t counts[2] = {scene->n_static, scene->n_dynamic};
    const char* names[2] = {"null static parameter", "null dynamic parameter"};
    for (int i = 0; i < 2; ++i) {
        const RdgSet& s = *sets[i];
        RDG_CHECK_ARG(counts[i] == 0 || (s.xyz && s.scaling && s.rotation && s.opacity && s.sh_dc &&
                                         (sh_degree == 0 || s.sh_rest)), names[i]);
        RDG_CHECK_ARG(counts[i] == 0 || (s.sh_dc_stride >= 3 && (sh_degree == 0 || s.sh_rest_stride >= 45)),
                      "SH stride too small (sh_dc_stride >= 3, sh_rest_stride >= 45)");
    }
    const bool deform = scene->use_deform && scene->n_dynamic > 0;
    if (deform) {
        RDG_CHECK_ARG(scene->num_basis > 0 && scene->num_basis <= RDG_NUM_BASIS_MAX, "num_basis out of range");
        RDG_CHECK_ARG(scene->num_times > 0, "num_times out of range");
        RDG_CHECK_ARG(scene->motion_coeff && scene->time_ind && scene->basis_t && scene->table, "null deformation input");
    }
    ExportParams p;
    p.sc = *scene;
    p.records = records;
    p.rest_coeffs = (sh_degree + 1) * (sh_degree + 1) - 1;
    p.diff_smem = 0;
    size_t smem = 0;
    if (deform && scene->num_basis == RDG_NUM_BASIS_MAX && scene->num_times <= RDG_EXPORT_TABLE_MAX &&
        (((uintptr_t)scene->basis_t | (uintptr_t)scene->table) & 15u) == 0) {
        p.diff_smem = 1;
        smem = (size_t)scene->num_times * RDG_DIFF_STRIDE * sizeof(float);
    }
    // persistent grid, so that each CTA stages the difference table once: 2 CTAs per SM (__launch_bounds__)
    const int64_t chunks = (scene->n_static + RDG_BLOCK - 1) / RDG_BLOCK + (scene->n_dynamic + RDG_BLOCK - 1) / RDG_BLOCK;
    const int grid = (int)(chunks < (int64_t)RDG_SM_COUNT * 2 ? chunks : (int64_t)RDG_SM_COUNT * 2);
    RDG_CUDA(cudaFuncSetAttribute(export_3dgs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    export_3dgs_kernel<<<grid, RDG_BLOCK, smem, (cudaStream_t)stream>>>(p);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}
