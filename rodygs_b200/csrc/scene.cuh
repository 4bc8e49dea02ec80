// Per-Gaussian parameter fetch shared by preprocess forward and backward:
// static||dynamic addressing without a concat, activations and the
// time-conditioned deformation, all in registers.
//
// Replaces, per Gaussian:
//   /root/reference/src/model/rodygs_static.py:82-105   (exp / normalize / sigmoid getters)
//   /root/reference/src/model/rodygs_dynamic.py:122-138 (c . (B(t) - B(t_i)), * spatial_lr_scale)
//   /root/reference/src/trainer/rodygs.py:68-113        (static first, dynamic second; delta-q added
//                                                        to the normalised quaternion, not re-normalised)
#pragma once
#include "common.cuh"
#include "tma.cuh"

struct RdgAct {
    float x, y, z;     // (deformed) mean
    float s[3];        // activated scale, before scale_modifier
    float q[4];        // quaternion as the rasterizer uses it (r,x,y,z)
    float op;          // opacity in [0,1]
    float qn[4];       // raw only: normalised raw quaternion
    float qinv;        // raw only: 1 / max(|raw|, 1e-12)
    float c[RDG_NUM_BASIS_MAX];  // dynamic only: motion coefficients
    int ti;            // dynamic only: birth-frame index
    bool dyn;
    int64_t local;     // index inside its own set
};

// B(t)[k][j] - table[ti][k][j].  B(t) is 112 floats that every thread reads at the same
// address (broadcast from shared memory or L1); the table row of the Gaussian's birth frame
// (448 B, 16-byte aligned) is read with vector loads and stays L1/L2 resident (T rows, 45 KB).
__device__ __forceinline__ float rdg_basis_diff(const RdgScene& sc, const float* basis_t, int ti, int k, int j) {
    return basis_t[k * 7 + j] - __ldg(sc.table + ((int64_t)ti * sc.num_basis + k) * 7 + j);
}

// Shared-memory copy of the differences B(t) - table[t'] for every frame t' (row stride RDG_DIFF_STRIDE floats).
// ncu r01: the per-lane gathers of 448-byte table rows (28 LDG.128 per dynamic Gaussian, 32 different rows per warp
// instruction = 32 L1 wavefronts each) kept the L1TEX pipe of both preprocess kernels 55-63 % busy - their top unit.  From
// shared memory the same row costs 28 LDS.128 at ~2 wavefronts each (116-float stride: 29 x 16 B, odd in 16-byte units,
// so the rows of the 8 lanes of a phase spread over all bank groups).
#define RDG_DIFF_STRIDE 116
// Only used with num_basis == RDG_NUM_BASIS_MAX: a row is 112 floats = 28 float4 (compile-time divisor).
__device__ __forceinline__ void rdg_stage_diff(const RdgScene& sc, const float* basis_t, float* diff_s, int nthreads) {
    const float4* tab4 = reinterpret_cast<const float4*>(sc.table);
    const float4* bt4 = reinterpret_cast<const float4*>(basis_t);
    for (int idx = threadIdx.x; idx < sc.num_times * 28; idx += nthreads) {
        const int t = idx / 28, q = idx - t * 28;
        const float4 b = __ldg(bt4 + q), r = __ldg(tab4 + idx);
        *reinterpret_cast<float4*>(diff_s + t * RDG_DIFF_STRIDE + 4 * q) = make_float4(b.x - r.x, b.y - r.y, b.z - r.z, b.w - r.w);
    }
}

// delta[j] = sum_k c_k (B(t)[k][j] - table[ti][k][j]),  j = 0..6.  diff_s: rdg_stage_diff()'s copy, or NULL (then the
// table row is gathered from global memory).  Same float operations either way: the results are bit-identical.
// The accumulation is an explicit fmaf chain: the deformed mean is an INPUT of the bit-exact part of the forward pass (the
// integer outputs are checked against the oracle run on the activated values the kernel itself produced), so it may be
// fused - 112 instructions instead of 224 per dynamic Gaussian in the -fmad=false forward translation unit.
__device__ __forceinline__ void rdg_deform_delta(const RdgScene& sc, const float* basis_t, int ti, const float* c, float* d,
                                                 const float* diff_s = nullptr) {
#pragma unroll
    for (int j = 0; j < 7; ++j) d[j] = 0.f;
    const float* row = sc.table + (int64_t)ti * sc.num_basis * 7;
    if (sc.num_basis == RDG_NUM_BASIS_MAX && diff_s) {
        const float4* row4 = reinterpret_cast<const float4*>(diff_s + ti * RDG_DIFF_STRIDE);
#pragma unroll
        for (int q = 0; q < 28; ++q) {
            const float4 v = row4[q];
            const float r[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const int e = 4 * q + m;
                d[e % 7] = fmaf(c[e / 7], r[m], d[e % 7]);   // explicit FMA: the forward TU is built with -fmad=false
            }
        }
    } else if (sc.num_basis == RDG_NUM_BASIS_MAX) {
        const float4* row4 = reinterpret_cast<const float4*>(row);   // 112 floats = 28 float4
#pragma unroll
        for (int q = 0; q < 28; ++q) {
            const float4 v = __ldg(row4 + q);
            const float r[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const int e = 4 * q + m;          // e = k*7 + j, compile-time after unrolling
                d[e % 7] = fmaf(c[e / 7], basis_t[e] - r[m], d[e % 7]);
            }
        }
    } else {
        for (int k = 0; k < sc.num_basis; ++k)
#pragma unroll
            for (int j = 0; j < 7; ++j) d[j] = fmaf(c[k], basis_t[k * 7 + j] - __ldg(row + k * 7 + j), d[j]);
    }
}

// delta[j] = sum_k c_k (B(t)[k][j] - table[ti][k][j]) from a table row staged in shared memory (stride RDG_DIFF_STRIDE,
// num_basis == RDG_NUM_BASIS_MAX) and B(t) kept apart: the batched forward stages the table once for all its views.  The
// difference is rounded on its own before the FMA, so the result has the bits of rdg_deform_delta's.
__device__ __forceinline__ void rdg_deform_delta_rows(const float* basis_t, const float* row_s, const float* c, float* d) {
#pragma unroll
    for (int j = 0; j < 7; ++j) d[j] = 0.f;
    const float4* row4 = reinterpret_cast<const float4*>(row_s);
    const float4* bt4 = reinterpret_cast<const float4*>(basis_t);
#pragma unroll
    for (int q = 0; q < 28; ++q) {
        const float4 v = row4[q], b = bt4[q];
        const float r[4] = {v.x, v.y, v.z, v.w}, bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            const int e = 4 * q + m;
            d[e % 7] = fmaf(c[e / 7], bb[m] - r[m], d[e % 7]);
        }
    }
}

// The deformation delta (rdg_deform_delta) applied to the activated parameters.
__device__ __forceinline__ void rdg_apply_deform(const RdgScene& sc, const float* d, RdgAct& a) {
    a.x += d[0] * sc.spatial_lr_scale;
    a.y += d[1] * sc.spatial_lr_scale;
    a.z += d[2] * sc.spatial_lr_scale;
    a.q[0] += d[3]; a.q[1] += d[4]; a.q[2] += d[5]; a.q[3] += d[6];
}

// Loads, activations and (DEFORM) the deformation of one Gaussian.  DEFORM = false stops at the canonical mean and
// quaternion and leaves a.c / a.ti loaded: the batched forward deforms each view's copy itself.
template <bool RAW, bool DEFORM = true>
__device__ __forceinline__ void rdg_fetch(const RdgScene& sc, bool dyn, int64_t local, const float* basis_t, RdgAct& a,
                                          const float* diff_s = nullptr) {
    a.dyn = dyn;
    a.local = local;
    const RdgSet& set = dyn ? sc.dy : sc.st;
    const float* px = set.xyz + local * 3;
    const float* ps = set.scaling + local * 3;
    const float4 q4 = __ldg(reinterpret_cast<const float4*>(set.rotation) + local);
    a.x = __ldg(px); a.y = __ldg(px + 1); a.z = __ldg(px + 2);
    const float s0 = __ldg(ps), s1 = __ldg(ps + 1), s2 = __ldg(ps + 2);
    const float q0 = q4.x, q1 = q4.y, q2 = q4.z, q3 = q4.w;
    const float o = __ldg(set.opacity + local);
    a.ti = 0;
    if (RAW) {
        a.s[0] = expf(s0); a.s[1] = expf(s1); a.s[2] = expf(s2);
        const float nrm = sqrtf(q0 * q0 + q1 * q1 + q2 * q2 + q3 * q3);
        a.qinv = 1.0f / fmaxf(nrm, 1e-12f);
        a.qn[0] = q0 * a.qinv; a.qn[1] = q1 * a.qinv; a.qn[2] = q2 * a.qinv; a.qn[3] = q3 * a.qinv;
        a.q[0] = a.qn[0]; a.q[1] = a.qn[1]; a.q[2] = a.qn[2]; a.q[3] = a.qn[3];
        a.op = 1.0f / (1.0f + expf(-o));
        if (dyn && sc.use_deform) {
            const float* pc = sc.motion_coeff + local * sc.num_basis;
            a.ti = __ldg(sc.time_ind + local);
            if (sc.num_basis == RDG_NUM_BASIS_MAX) {
                const float4* pc4 = reinterpret_cast<const float4*>(pc);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 v = __ldg(pc4 + q);
                    a.c[4 * q] = v.x; a.c[4 * q + 1] = v.y; a.c[4 * q + 2] = v.z; a.c[4 * q + 3] = v.w;
                }
            } else {
#pragma unroll
                for (int k = 0; k < RDG_NUM_BASIS_MAX; ++k) a.c[k] = k < sc.num_basis ? __ldg(pc + k) : 0.f;
            }
            if (DEFORM) {
                float d[7];
                rdg_deform_delta(sc, basis_t, a.ti, a.c, d, diff_s);
                rdg_apply_deform(sc, d, a);
            }
        }
    } else {
        a.s[0] = s0; a.s[1] = s1; a.s[2] = s2;
        a.q[0] = q0; a.q[1] = q1; a.q[2] = q2; a.q[3] = q3;
        a.qn[0] = q0; a.qn[1] = q1; a.qn[2] = q2; a.qn[3] = q3;
        a.qinv = 1.0f;
        a.op = o;
    }
}

// L2 prefetch (rdg_bulk_prefetch_l2, tma.cuh) of the parameter rows of 256-Gaussian chunk `chunk`: thread f = 0..7 of the CTA
// takes one field.  cs = number of static chunks.  acc: the blend backward's accumulator rows (backward pass) or NULL.
__device__ __forceinline__ void rdg_prefetch_chunk_field(const RdgScene& sc, int64_t chunk, int64_t cs, int f, const float* acc) {
    const bool dyn = chunk >= cs;
    const RdgSet& set = dyn ? sc.dy : sc.st;
    const int64_t lbase = (dyn ? chunk - cs : chunk) * RDG_BLOCK;
    const int64_t n_set = dyn ? sc.n_dynamic : sc.n_static;
    const int64_t cnt = min((int64_t)RDG_BLOCK, n_set - lbase);
    if (cnt <= 0) return;
    const char* ptr = nullptr;
    int64_t bytes = 0;
    switch (f) {
        case 0: ptr = (const char*)(set.xyz + lbase * 3); bytes = cnt * 12; break;
        case 1: ptr = (const char*)(set.scaling + lbase * 3); bytes = cnt * 12; break;
        case 2: ptr = (const char*)(set.rotation + lbase * 4); bytes = cnt * 16; break;
        case 3: ptr = (const char*)(set.opacity + lbase); bytes = cnt * 4; break;
        case 4: if (set.sh_dc && set.sh_dc_stride == 3) { ptr = (const char*)(set.sh_dc + lbase * 3); bytes = cnt * 12; } break;
        case 5: if (acc) { ptr = (const char*)(acc + ((dyn ? sc.n_static : 0) + lbase) * 12); bytes = cnt * 48; } break;
        case 6: if (dyn && sc.raw && sc.use_deform && sc.motion_coeff) { ptr = (const char*)(sc.motion_coeff + lbase * sc.num_basis); bytes = cnt * sc.num_basis * 4; } break;
        default: if (dyn && sc.raw && sc.use_deform && sc.time_ind) { ptr = (const char*)(sc.time_ind + lbase); bytes = cnt * 4; } break;
    }
    bytes &= ~(int64_t)15;
    if (ptr && bytes > 0 && ((uintptr_t)ptr & 15u) == 0) rdg_bulk_prefetch_l2(ptr, (uint32_t)bytes);
}

// Everything downstream of the activated parameters that both passes need.
struct RdgProj {
    float tx, ty, tz;          // view-space mean
    float hx, hy, hw, pw;      // clip space and 1/(w+1e-7)
    float R[9];                // rotation from the quaternion (row-major)
    float M[9];                // R * diag(s * scale_modifier)
    float S[6];                // Sigma: 00 01 02 11 12 22
    float ctx, cty;            // clamped t.x, t.y used in J
    bool in_x, in_y;
    float J00, J02, J11, J12;
    float T[6];                // J*W: T00 T01 T02 T10 T11 T12
    float ca, cb, cc;          // 2D covariance after the low-pass
    float det;
};

// App. A.2 steps 1-5 in the exact operation order of oracle/splat_oracle.py
// (the forward translation unit is compiled with -fmad=false).
__device__ __forceinline__ void rdg_project(const RdgCam& cam, const RdgAct& a, float scale_modifier, RdgProj& p) {
    const float* V = cam.V;
    const float* P = cam.P;
    p.tx = V[0] * a.x + V[1] * a.y + V[2] * a.z + V[3];
    p.ty = V[4] * a.x + V[5] * a.y + V[6] * a.z + V[7];
    p.tz = V[8] * a.x + V[9] * a.y + V[10] * a.z + V[11];
    p.hx = P[0] * p.tx + P[1] * p.ty + P[2] * p.tz + P[3];
    p.hy = P[4] * p.tx + P[5] * p.ty + P[6] * p.tz + P[7];
    p.hw = P[12] * p.tx + P[13] * p.ty + P[14] * p.tz + P[15];
    p.pw = 1.0f / (p.hw + 0.0000001f);

    const float qr = a.q[0], qx = a.q[1], qy = a.q[2], qz = a.q[3];
    p.R[0] = 1.0f - 2.0f * (qy * qy + qz * qz);
    p.R[1] = 2.0f * (qx * qy - qr * qz);
    p.R[2] = 2.0f * (qx * qz + qr * qy);
    p.R[3] = 2.0f * (qx * qy + qr * qz);
    p.R[4] = 1.0f - 2.0f * (qx * qx + qz * qz);
    p.R[5] = 2.0f * (qy * qz - qr * qx);
    p.R[6] = 2.0f * (qx * qz - qr * qy);
    p.R[7] = 2.0f * (qy * qz + qr * qx);
    p.R[8] = 1.0f - 2.0f * (qx * qx + qy * qy);
    const float s0 = a.s[0] * scale_modifier, s1 = a.s[1] * scale_modifier, s2 = a.s[2] * scale_modifier;
    float* M = p.M;
    M[0] = p.R[0] * s0; M[1] = p.R[1] * s1; M[2] = p.R[2] * s2;
    M[3] = p.R[3] * s0; M[4] = p.R[4] * s1; M[5] = p.R[5] * s2;
    M[6] = p.R[6] * s0; M[7] = p.R[7] * s1; M[8] = p.R[8] * s2;
    p.S[0] = M[0] * M[0] + M[1] * M[1] + M[2] * M[2];
    p.S[1] = M[0] * M[3] + M[1] * M[4] + M[2] * M[5];
    p.S[2] = M[0] * M[6] + M[1] * M[7] + M[2] * M[8];
    p.S[3] = M[3] * M[3] + M[4] * M[4] + M[5] * M[5];
    p.S[4] = M[3] * M[6] + M[4] * M[7] + M[5] * M[8];
    p.S[5] = M[6] * M[6] + M[7] * M[7] + M[8] * M[8];

    const float txtz = p.tx / p.tz;
    const float tytz = p.ty / p.tz;
    p.in_x = (txtz >= -cam.limx) && (txtz <= cam.limx);
    p.in_y = (tytz >= -cam.limy) && (tytz <= cam.limy);
    p.ctx = fminf(cam.limx, fmaxf(-cam.limx, txtz)) * p.tz;
    p.cty = fminf(cam.limy, fmaxf(-cam.limy, tytz)) * p.tz;
    const float tz2 = p.tz * p.tz;
    p.J00 = cam.fx / p.tz;
    p.J02 = -(cam.fx * p.ctx) / tz2;
    p.J11 = cam.fy / p.tz;
    p.J12 = -(cam.fy * p.cty) / tz2;
    float* T = p.T;
    T[0] = p.J00 * V[0] + p.J02 * V[8];
    T[1] = p.J00 * V[1] + p.J02 * V[9];
    T[2] = p.J00 * V[2] + p.J02 * V[10];
    T[3] = p.J11 * V[4] + p.J12 * V[8];
    T[4] = p.J11 * V[5] + p.J12 * V[9];
    T[5] = p.J11 * V[6] + p.J12 * V[10];
    const float* S = p.S;
    const float U00 = T[0] * S[0] + T[1] * S[1] + T[2] * S[2];
    const float U01 = T[0] * S[1] + T[1] * S[3] + T[2] * S[4];
    const float U02 = T[0] * S[2] + T[1] * S[4] + T[2] * S[5];
    const float U10 = T[3] * S[0] + T[4] * S[1] + T[5] * S[2];
    const float U11 = T[3] * S[1] + T[4] * S[3] + T[5] * S[4];
    const float U12 = T[3] * S[2] + T[4] * S[4] + T[5] * S[5];
    p.ca = U00 * T[0] + U01 * T[1] + U02 * T[2] + RDG_LOWPASS;
    p.cb = U00 * T[3] + U01 * T[4] + U02 * T[5];
    p.cc = U10 * T[3] + U11 * T[4] + U12 * T[5] + RDG_LOWPASS;
    p.det = p.ca * p.cc - p.cb * p.cb;
}

// SH basis values for a unit direction (sh_utils.py:72-101), b[0..K-1].
template <int deg>
__device__ __forceinline__ void rdg_sh_basis(float x, float y, float z, float* b) {
    b[0] = RDG_SH_C0;
    if (deg > 0) {
        b[1] = -RDG_SH_C1 * y;
        b[2] = RDG_SH_C1 * z;
        b[3] = -RDG_SH_C1 * x;
        if (deg > 1) {
            float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
            b[4] = RDG_SH_C2_0 * xy;
            b[5] = RDG_SH_C2_1 * yz;
            b[6] = RDG_SH_C2_2 * (2.0f * zz - xx - yy);
            b[7] = RDG_SH_C2_3 * xz;
            b[8] = RDG_SH_C2_4 * (xx - yy);
            if (deg > 2) {
                b[9] = RDG_SH_C3_0 * y * (3.0f * xx - yy);
                b[10] = RDG_SH_C3_1 * xy * z;
                b[11] = RDG_SH_C3_2 * y * (4.0f * zz - xx - yy);
                b[12] = RDG_SH_C3_3 * z * (2.0f * zz - 3.0f * xx - 3.0f * yy);
                b[13] = RDG_SH_C3_4 * x * (4.0f * zz - xx - yy);
                b[14] = RDG_SH_C3_5 * z * (xx - yy);
                b[15] = RDG_SH_C3_6 * x * (xx - 3.0f * yy);
            }
        }
    }
}

// camera position  -R^T T  from the unpacked view matrix
__device__ __forceinline__ void rdg_campos(const RdgCam& cam, float* cp) {
    const float* V = cam.V;
    cp[0] = -(V[0] * V[3] + V[4] * V[7] + V[8] * V[11]);
    cp[1] = -(V[1] * V[3] + V[5] * V[7] + V[9] * V[11]);
    cp[2] = -(V[2] * V[3] + V[6] * V[7] + V[10] * V[11]);
}
