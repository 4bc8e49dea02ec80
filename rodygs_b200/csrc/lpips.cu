// LPIPS (the lpips package v0.1, lpips=True, spatial=False) of a batch of image pairs with the AlexNet or VGG-16 backbone,
// from the user's weight files (INTEGRATION.md "Scoring held-out views").  Pairs are processed in turn through one pair's
// workspace; per pair:
//   scale       pred, gt [3, H, W] -> x' = (x / R - mu) / sigma, NHWC [2][H][W][3] (image 0 = pred, 1 = gt)
//   conv        conv + bias + ReLU as an implicit GEMM on tcgen05 tensor cores (kind::tf32, FP32 accumulators in TMEM)
//   pool        max-pool k3 s2 (alex) / k2 s2 (vgg), floor, NHWC
//   head        after each of the five taps: per position sum_c w_c (f0_c / |f0| - f1_c / |f1|)^2 -> per-CTA float64 slots
//   finalize    one CTA: sum over taps of (sum of the tap's slots in a fixed order) / positions
// Activations ping-pong between two NHWC buffers; the head runs straight after its tap, so a tap's features are dead before
// the next layer overwrites them.  No float atomics: bit-identical from run to run and independent of the rest of the batch.
//
// Masked LPIPS (rdg_masked_lpips, DyCheck's mLPIPS) runs the same pass with three changes:
//   scale       x_m = m != 0 ? m x : 0 before the scaling, likewise y_m
//   head        writes sum_c w_c (...)^2 of every position as float32 to the tap's map in the workspace instead of summing it
//   spatial     one pass over the H x W pixels: sum over taps of the bilinear upsample (align_corners=False) of each map,
//               weighted by m, into per-CTA float64 slots of sum m map and sum m; a one-CTA finalize divides the two
//
// Conv GEMM: M = output pixels of both images, N = Cout, K = kh kw Cin ordered (ky, kx, c), so that with NHWC activations a
// 32-wide K slice is a contiguous run of channels of one input pixel (every Cin but the first layer's 3 is a multiple of 32;
// the first layer gathers element-wise and its K is zero-padded to a multiple of 32).  A CTA computes a 128 x BN tile:
//   warps 0-3   gather the A tile (im2col on the fly) into shared memory in the no-swizzle K-major core-matrix layout
//               (8 rows x 16 bytes per core matrix), rounding to TF32 with cvt.rna (round to nearest, ties away from zero);
//               thread 0 also bulk-copies the stage's B tile, which rdg_lpips_pack stored in the same layout, already rounded.
//               Afterwards they are the epilogue: tcgen05.ld of their 32 TMEM lanes, + bias, ReLU, NHWC store.
//   warp 4      allocates the TMEM accumulator, issues tcgen05.mma (one thread) and frees each stage with tcgen05.commit.
// Both operands are exact TF32 values, so the tensor core's handling of the low mantissa bits does not matter.
#include <math.h>
#include "common.cuh"
#include "tma.cuh"

#define LP_BM 128                    // output pixels per CTA (MMA M; TMEM lane = tile row)
#define LP_BK 32                     // K per stage (4 MMAs of K = 8)
#define LP_STAGES 3
#define LP_THREADS 160               // 4 gather / epilogue warps + the MMA warp
#define LP_A_CHUNK (LP_BM * 16 + 64) // bytes between the 8 core-matrix columns of an A stage (+64: conflict-free stores)
#define LP_A_STAGE (8 * LP_A_CHUNK)
#define LP_MAX_BN 128
#define LP_B_STAGE (LP_MAX_BN * LP_BK * 4)
#define LP_HEAD_THREADS 256
#define LP_HEAD_MAX_CTAS 1184        // 8 x 148
#define LP_TAPS 5
#define LP_MAX_LAYERS 18
#define LP_SPATIAL_THREADS 256
#define LP_SPATIAL_MAX_CTAS 1184     // 8 x 148

// ---- network definitions -----------------------------------------------------------------------------------------------

struct LpLayer {
    int conv;            // 1 conv + ReLU, 0 max-pool
    int cin, cout, k, s, p;
    int tap;             // a conv whose ReLU output is one of the five taps
};

static const LpLayer kAlex[] = {
    {1, 3, 64, 11, 4, 2, 1},    {0, 64, 64, 3, 2, 0, 0},     {1, 64, 192, 5, 1, 2, 1},   {0, 192, 192, 3, 2, 0, 0},
    {1, 192, 384, 3, 1, 1, 1},  {1, 384, 256, 3, 1, 1, 1},   {1, 256, 256, 3, 1, 1, 1},
};
static const LpLayer kVgg[] = {
    {1, 3, 64, 3, 1, 1, 0},     {1, 64, 64, 3, 1, 1, 1},     {0, 64, 64, 2, 2, 0, 0},
    {1, 64, 128, 3, 1, 1, 0},   {1, 128, 128, 3, 1, 1, 1},   {0, 128, 128, 2, 2, 0, 0},
    {1, 128, 256, 3, 1, 1, 0},  {1, 256, 256, 3, 1, 1, 0},   {1, 256, 256, 3, 1, 1, 1},   {0, 256, 256, 2, 2, 0, 0},
    {1, 256, 512, 3, 1, 1, 0},  {1, 512, 512, 3, 1, 1, 0},   {1, 512, 512, 3, 1, 1, 1},   {0, 512, 512, 2, 2, 0, 0},
    {1, 512, 512, 3, 1, 1, 0},  {1, 512, 512, 3, 1, 1, 0},   {1, 512, 512, 3, 1, 1, 1},
};

struct LpNet {
    const LpLayer* layers;
    int n;
    int min_edge;
};

static bool lp_net(int32_t net, LpNet* N) {
    if (net == RDG_LPIPS_ALEX) { *N = {kAlex, (int)(sizeof(kAlex) / sizeof(kAlex[0])), 31}; return true; }
    if (net == RDG_LPIPS_VGG) { *N = {kVgg, (int)(sizeof(kVgg) / sizeof(kVgg[0])), 16}; return true; }
    return false;
}

static int lp_bn(int cout) { return cout % 128 == 0 ? 128 : 64; }
static int lp_kpad(const LpLayer& L) { return (int)rdg_align_up((int64_t)L.k * L.k * L.cin, LP_BK); }

// Packed weights: per conv, in order, [Cout / BN][Kpad / 32][8][BN][4] TF32-rounded floats (the B stages), then bias [Cout];
// after the convs the five linear heads [C_l].  Every block starts on a 16-byte boundary.
struct LpPacked {
    int64_t w_off[LP_MAX_LAYERS], b_off[LP_MAX_LAYERS], lin_off[LP_TAPS];
    int64_t total;
};

static void lp_packed_layout(const LpNet& N, LpPacked* P) {
    int64_t off = 0;
    int t = 0;
    for (int i = 0; i < N.n; ++i) {
        const LpLayer& L = N.layers[i];
        if (!L.conv) continue;
        P->w_off[i] = off;
        off += (int64_t)L.cout * lp_kpad(L);
        P->b_off[i] = off;
        off += rdg_align_up(L.cout, 4);
    }
    for (int i = 0; i < N.n; ++i)
        if (N.layers[i].conv && N.layers[i].tap) {
            P->lin_off[t++] = off;
            off += rdg_align_up(N.layers[i].cout, 4);
        }
    P->total = off;
}

// Workspace of one pair: two activation buffers (the largest NHWC tensor of the pass, both images), then the head slots;
// masked, the five tap maps and the spatial pass's slots instead of the head slots.
struct LpWork {
    int64_t act_bytes;
    int64_t part_off[LP_TAPS];   // unmasked: [head_ctas] float64 per tap
    int head_ctas[LP_TAPS];
    int tap_h[LP_TAPS], tap_w[LP_TAPS];
    int64_t map_off[LP_TAPS];    // masked: [tap_h][tap_w] float32 per tap
    int64_t spatial_off;         // masked: [2][spatial_ctas] float64 (sum m map, then sum m)
    int spatial_ctas;
    int64_t total;
};

static int lp_head_ctas(int64_t positions) {
    const int64_t need = (positions + LP_HEAD_THREADS / 32 - 1) / (LP_HEAD_THREADS / 32);
    return (int)(need < LP_HEAD_MAX_CTAS ? need : LP_HEAD_MAX_CTAS);
}

static void lp_work_layout(const LpNet& N, int H, int W, bool masked, LpWork* Wk) {
    int64_t big = 2LL * H * W * 3;
    int h = H, w = W, t = 0;
    for (int i = 0; i < N.n; ++i) {
        const LpLayer& L = N.layers[i];
        h = (h + 2 * L.p - L.k) / L.s + 1;
        w = (w + 2 * L.p - L.k) / L.s + 1;
        const int64_t n = 2LL * h * w * L.cout;
        if (n > big) big = n;
        if (L.conv && L.tap) {
            Wk->tap_h[t] = h;
            Wk->tap_w[t] = w;
            ++t;
        }
    }
    Wk->act_bytes = rdg_align_up(big * (int64_t)sizeof(float), 256);
    int64_t off = 2 * Wk->act_bytes;
    for (int i = 0; i < LP_TAPS; ++i) {
        const int64_t positions = (int64_t)Wk->tap_h[i] * Wk->tap_w[i];
        Wk->head_ctas[i] = lp_head_ctas(positions);
        if (masked) {
            Wk->map_off[i] = off;
            off += rdg_align_up(positions * (int64_t)sizeof(float), 256);
        } else {
            Wk->part_off[i] = off;
            off += rdg_align_up((int64_t)Wk->head_ctas[i] * (int64_t)sizeof(double), 256);
        }
    }
    if (masked) {
        const int64_t need = ((int64_t)H * W + LP_SPATIAL_THREADS - 1) / LP_SPATIAL_THREADS;
        Wk->spatial_ctas = (int)(need < LP_SPATIAL_MAX_CTAS ? need : LP_SPATIAL_MAX_CTAS);
        Wk->spatial_off = off;
        off += rdg_align_up(2LL * Wk->spatial_ctas * (int64_t)sizeof(double), 256);
    }
    Wk->total = off;
}

// ---- device helpers ----------------------------------------------------------------------------------------------------

__device__ __forceinline__ uint32_t lp_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}

__device__ __forceinline__ void lp_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(rdg_smem_addr(bar)) : "memory");
}

// Shared-memory matrix descriptor, no swizzle, K-major: LBO = bytes between core matrices along K, SBO = bytes between
// 8-row groups along M / N; bits 46-47 = 1 (the sm_100 descriptor version).
__device__ __forceinline__ uint64_t lp_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}

// ---- conv + bias + ReLU ------------------------------------------------------------------------------------------------

struct LpConv {
    const float* in;     // NHWC [2][H][W][cin]
    float* out;          // NHWC [2][Ho][Wo][cout]
    const float* wpk;    // packed B stages of this layer
    const float* bias;   // [cout]
    int H, W, cin, Ho, Wo, cout, k, s, p;
    int M, kchunks, bn, ntiles;
};

__global__ void __launch_bounds__(LP_THREADS) lpips_conv_kernel(const LpConv c) {
    extern __shared__ __align__(1024) unsigned char lp_smem[];
    unsigned char* sA = lp_smem;                                   // [stages][LP_A_STAGE]
    unsigned char* sB = lp_smem + LP_STAGES * LP_A_STAGE;          // [stages][LP_B_STAGE]
    uint64_t* full = reinterpret_cast<uint64_t*>(sB + LP_STAGES * LP_B_STAGE);
    uint64_t* empty = full + LP_STAGES;
    uint64_t* done = empty + LP_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int mt = blockIdx.x / c.ntiles, nt = blockIdx.x - mt * c.ntiles;
    const int m0 = mt * LP_BM, n0 = nt * c.bn;
    const uint32_t b_bytes = (uint32_t)c.bn * LP_BK * 4;

    if (threadIdx.x == 0) {
        for (int s = 0; s < LP_STAGES; ++s) {
            rdg_mbar_init(&full[s], 4 * 32 + 1);   // every gather thread + the expect_tx of the B copy
            rdg_mbar_init(&empty[s], 1);           // tcgen05.commit
        }
        rdg_mbar_init(done, 1);
    }
    if (warp == 4) {
        // c.bn columns (64 or 128, a power of two >= 32); two CTAs per SM use at most 256 of the 512
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(rdg_smem_addr(tmem_slot)),
                     "r"((uint32_t)c.bn)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;

    if (warp < 4) {
        // ---- gather: thread -> float4 column q of rows r0 + 16 i ----
        const int t = threadIdx.x, q = t & 7, r0 = t >> 3;
        const int hw = c.Ho * c.Wo;
        int by[8], bx[8];
        int64_t base[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int m = m0 + r0 + 16 * i;
            if (m < c.M) {
                const int img = m / hw, rem = m - img * hw, oy = rem / c.Wo, ox = rem - oy * c.Wo;
                by[i] = oy * c.s - c.p;
                bx[i] = ox * c.s - c.p;
                base[i] = (int64_t)img * c.H * c.W;
            } else {
                by[i] = -(1 << 20);   // every tap out of bounds: a zero row
                bx[i] = 0;
                base[i] = 0;
            }
        }
        const bool vec = (c.cin % LP_BK) == 0;
        const int kreal = c.k * c.k * c.cin;
        for (int kc = 0; kc < c.kchunks; ++kc) {
            const int s = kc % LP_STAGES;
            if (kc >= LP_STAGES) rdg_mbar_wait(&empty[s], ((kc / LP_STAGES) - 1) & 1);
            if (t == 0)
                rdg_bulk_load(sB + s * LP_B_STAGE, c.wpk + ((int64_t)nt * c.kchunks + kc) * c.bn * LP_BK, b_bytes, &full[s]);
            unsigned char* a = sA + s * LP_A_STAGE + q * LP_A_CHUNK;
            if (vec) {
                const int k0 = kc * LP_BK, tap = k0 / c.cin, c0 = k0 - tap * c.cin;
                const int ky = tap / c.k, kx = tap - ky * c.k;
                float4 v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int iy = by[i] + ky, ix = bx[i] + kx;
                    v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (iy >= 0 && iy < c.H && ix >= 0 && ix < c.W)
                        v[i] = __ldg(reinterpret_cast<const float4*>(c.in + (base[i] + (int64_t)iy * c.W + ix) * c.cin + c0) + q);
                }
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    *reinterpret_cast<uint4*>(a + (r0 + 16 * i) * 16) =
                        make_uint4(lp_tf32(v[i].x), lp_tf32(v[i].y), lp_tf32(v[i].z), lp_tf32(v[i].w));
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    uint32_t e[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int kk = kc * LP_BK + q * 4 + j;
                        float v = 0.f;
                        if (kk < kreal) {
                            const int tap = kk / c.cin, ch = kk - tap * c.cin, ky = tap / c.k, kx = tap - ky * c.k;
                            const int iy = by[i] + ky, ix = bx[i] + kx;
                            if (iy >= 0 && iy < c.H && ix >= 0 && ix < c.W)
                                v = __ldg(c.in + (base[i] + (int64_t)iy * c.W + ix) * c.cin + ch);
                        }
                        e[j] = lp_tf32(v);
                    }
                    *reinterpret_cast<uint4*>(a + (r0 + 16 * i) * 16) = make_uint4(e[0], e[1], e[2], e[3]);
                }
            }
            rdg_fence_proxy_async();   // the generic-proxy stores above, before the tensor core reads them
            lp_mbar_arrive(&full[s]);
        }
        // ---- epilogue: TMEM lanes 32 warp .. 32 warp + 31 = tile rows ----
        rdg_mbar_wait(done, 0);
        __syncwarp();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int m = m0 + warp * 32 + lane;
        float* orow = c.out + (int64_t)m * c.cout + n0;
        for (int j = 0; j < c.bn; j += 16) {
            uint32_t r[16];
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                  "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                : "r"(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)j));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (m < c.M) {
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const float4 b = __ldg(reinterpret_cast<const float4*>(c.bias + n0 + j) + g);
                    float4 o;
                    o.x = fmaxf(__uint_as_float(r[4 * g + 0]) + b.x, 0.f);
                    o.y = fmaxf(__uint_as_float(r[4 * g + 1]) + b.y, 0.f);
                    o.z = fmaxf(__uint_as_float(r[4 * g + 2]) + b.z, 0.f);
                    o.w = fmaxf(__uint_as_float(r[4 * g + 3]) + b.w, 0.f);
                    reinterpret_cast<float4*>(orow + j)[g] = o;
                }
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    } else if (lane == 0) {
        // ---- MMA issue: D[128 x bn] (+)= A[128 x 8] B[8 x bn]^T, four per stage ----
        const uint32_t idesc = (1u << 4)                     // D: f32
                               | (2u << 7) | (2u << 10)      // A, B: tf32; both K-major, no negation
                               | ((uint32_t)(c.bn >> 3) << 17) | ((uint32_t)(LP_BM >> 4) << 24);
        const uint32_t b_chunk = (uint32_t)c.bn * 16;
        for (int kc = 0; kc < c.kchunks; ++kc) {
            const int s = kc % LP_STAGES;
            rdg_mbar_wait(&full[s], (kc / LP_STAGES) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t a0 = rdg_smem_addr(sA + s * LP_A_STAGE), b0 = rdg_smem_addr(sB + s * LP_B_STAGE);
#pragma unroll
            for (int j = 0; j < LP_BK / 8; ++j) {
                const uint64_t ad = lp_desc(a0 + 2 * j * LP_A_CHUNK, LP_A_CHUNK, 128);
                const uint64_t bd = lp_desc(b0 + 2 * j * b_chunk, b_chunk, 128);
                const uint32_t acc = (kc > 0 || j > 0) ? 1u : 0u;
                asm volatile(
                    "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                    "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem),
                    "l"(ad), "l"(bd), "r"(idesc), "r"(acc)
                    : "memory");
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                             rdg_smem_addr(&empty[s]))
                         : "memory");
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(rdg_smem_addr(done))
                     : "memory");
    }
    __syncthreads();
    if (warp == 4) {
        __syncwarp();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)c.bn) : "memory");
    }
}

static const size_t kConvSmem = (size_t)LP_STAGES * (LP_A_STAGE + LP_B_STAGE) + (2 * LP_STAGES + 1) * 8 + 16;

// ---- weights packing ---------------------------------------------------------------------------------------------------

// w [cout, cin, k, k] (torch) -> [cout / bn][kpad / 32][8][bn][4], element (kc, q, n, e) = W[nt bn + n] at K index
// kc 32 + 4 q + e = (ky k + kx) cin + c, rounded to TF32 (rna); 0 past the real K
__global__ void lpips_pack_kernel(const float* __restrict__ w, float* __restrict__ dst, int cin, int cout, int k, int kpad,
                                  int bn) {
    const int64_t n_all = (int64_t)cout * kpad;
    const int kreal = k * k * cin, kchunks = kpad / LP_BK;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_all; i += (int64_t)gridDim.x * blockDim.x) {
        const int e = (int)(i & 3);
        int64_t r = i >> 2;
        const int n = (int)(r % bn);
        r /= bn;
        const int q = (int)(r & 7);
        r >>= 3;
        const int kc = (int)(r % kchunks), nt = (int)(r / kchunks);
        const int kk = kc * LP_BK + q * 4 + e, co = nt * bn + n;
        float v = 0.f;
        if (kk < kreal) {
            const int tap = kk / cin, ch = kk - tap * cin, ky = tap / k, kx = tap - ky * k;
            v = w[(((int64_t)co * cin + ch) * k + ky) * k + kx];
        }
        dst[i] = __uint_as_float(lp_tf32(v));
    }
}

__global__ void lpips_copy_kernel(const float* __restrict__ src, float* __restrict__ dst, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[i];
}

// ---- scaling, pooling, head, finalize ----------------------------------------------------------------------------------

// pred, gt [3, H, W] -> out NHWC [2][H][W][3], (x / R - mu_c) / sigma_c; with a mask [H, W] (NULL: none), x is first
// replaced by m != 0 ? m x : 0, so values under m = 0 take no part, NaN included
__global__ void lpips_scale_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                   const float* __restrict__ mask, int H, int W, float R, float* __restrict__ out) {
    const int64_t hw = (int64_t)H * W;
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= 2 * hw) return;
    const float* src = i < hw ? pred : gt;
    const int64_t p = i < hw ? i : i - hw;
    const float m = mask ? mask[p] : 1.f;
    const float mu[3] = {0.485f, 0.456f, 0.406f}, sd[3] = {0.229f, 0.224f, 0.225f};
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        float v = src[ch * hw + p];
        if (mask) v = m != 0.f ? m * v : 0.f;
        out[i * 3 + ch] = (v / R - mu[ch]) / sd[ch];
    }
}

// NHWC [2][H][W][C] -> [2][Ho][Wo][C], window k, stride s, no padding, floor
__global__ void lpips_pool_kernel(const float4* __restrict__ in, float4* __restrict__ out, int H, int W, int C4, int Ho, int Wo,
                                  int k, int s) {
    const int64_t n = 2LL * Ho * Wo * C4;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C4);
        int64_t r = i / C4;
        const int ox = (int)(r % Wo);
        r /= Wo;
        const int oy = (int)(r % Ho), img = (int)(r / Ho);
        const float4* src = in + (((int64_t)img * H + oy * s) * W + ox * s) * C4 + c;
        float4 m = src[0];
        for (int dy = 0; dy < k; ++dy)
            for (int dx = 0; dx < k; ++dx) {
                const float4 v = src[((int64_t)dy * W + dx) * C4];
                m.x = fmaxf(m.x, v.x);
                m.y = fmaxf(m.y, v.y);
                m.z = fmaxf(m.z, v.z);
                m.w = fmaxf(m.w, v.w);
            }
        out[i] = m;
    }
}

__device__ __forceinline__ float lp_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// f NHWC [2][positions][C] (C a multiple of 32, <= 512), one warp per position, d[p] = sum_c w_c (f0_c / (|f0| + 1e-10) -
// f1_c / (|f1| + 1e-10))^2:  part[blockIdx.x] = sum over the CTA's positions of d[p]; MAP: map[p] = d[p] (part unused)
template <bool MAP>
__global__ void __launch_bounds__(LP_HEAD_THREADS) lpips_head_kernel(const float* __restrict__ f, const float* __restrict__ lin,
                                                                     int64_t positions, int C, double* __restrict__ part,
                                                                     float* __restrict__ map) {
    __shared__ double red[LP_HEAD_THREADS / 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, per = C / 32;
    double acc = 0.0;
    for (int64_t p = (int64_t)blockIdx.x * (LP_HEAD_THREADS / 32) + warp; p < positions;
         p += (int64_t)gridDim.x * (LP_HEAD_THREADS / 32)) {
        const float* a = f + p * C;
        const float* b = f + (positions + p) * C;
        float va[16], vb[16], sa = 0.f, sb = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            va[i] = vb[i] = 0.f;
            if (i < per) {
                va[i] = a[lane + 32 * i];
                vb[i] = b[lane + 32 * i];
                sa = fmaf(va[i], va[i], sa);
                sb = fmaf(vb[i], vb[i], sb);
            }
        }
        const float na = sqrtf(lp_warp_sum(sa)) + 1e-10f, nb = sqrtf(lp_warp_sum(sb)) + 1e-10f;
        float d = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (i < per) {
                const float diff = va[i] / na - vb[i] / nb;
                d = fmaf(lin[lane + 32 * i], diff * diff, d);
            }
        const float dp = lp_warp_sum(d);
        if constexpr (MAP) {
            if (lane == 0) map[p] = dp;
        } else {
            acc += (double)dp;
        }
    }
    if constexpr (!MAP) {
        if (lane == 0) red[warp] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < LP_HEAD_THREADS / 32; ++w) t += red[w];
            part[blockIdx.x] = t;
        }
    }
}

struct LpFinal {
    const double* part[LP_TAPS];
    int ctas[LP_TAPS];
    double positions[LP_TAPS];
};

__global__ void __launch_bounds__(256) lpips_finalize_kernel(LpFinal fin, float* __restrict__ out) {
    __shared__ double sh[256];
    double total = 0.0;
    for (int l = 0; l < LP_TAPS; ++l) {
        double t = 0.0;
        for (int i = threadIdx.x; i < fin.ctas[l]; i += 256) t += fin.part[l][i];
        sh[threadIdx.x] = t;
        __syncthreads();
        for (int s = 128; s > 0; s >>= 1) {
            if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
            __syncthreads();
        }
        total += sh[0] / fin.positions[l];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = (float)total;
}

struct LpSpatial {
    const float* map[LP_TAPS];       // [h][w] float32
    int h[LP_TAPS], w[LP_TAPS];
    float sy[LP_TAPS], sx[LP_TAPS];  // in / out per axis, divided in float32 as ATen does for float32 input
};

// One axis of nn.Upsample(mode="bilinear", align_corners=False): src = max(scale (dst + 0.5) - 0.5, 0), taps i0 = floor(src)
// and i1 = min(i0 + 1, in - 1) with weights 1 - l1 and l1 = src - i0
__device__ __forceinline__ void lp_bilinear_axis(float scale, int dst, int in, int* i0, int* i1, float* l1) {
    const float src = fmaxf(scale * ((float)dst + 0.5f) - 0.5f, 0.f);
    *i0 = (int)src;   // src >= 0: truncation is floor
    *i1 = *i0 < in - 1 ? *i0 + 1 : *i0;
    *l1 = src - (float)*i0;
}

// mask [H][W]: part[blockIdx.x] = sum over the CTA's pixels of m map, part[gridDim.x + blockIdx.x] = sum of m, with map the
// float32 sum over taps (in tap order) of each upsampled tap map.  Pixels with m = 0 are skipped: they add nothing to either
// sum.  Fixed pixel-to-thread assignment and a fixed-order reduction: no atomics.
__global__ void __launch_bounds__(LP_SPATIAL_THREADS) lpips_spatial_kernel(const LpSpatial sp, const float* __restrict__ mask,
                                                                           int H, int W, double* __restrict__ part) {
    __shared__ double red[2][LP_SPATIAL_THREADS / 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int hw = H * W;   // <= 2^26 (lp_check_size): 32-bit pixel indices
    double am = 0.0, an = 0.0;
    for (int p = blockIdx.x * LP_SPATIAL_THREADS + threadIdx.x; p < hw; p += gridDim.x * LP_SPATIAL_THREADS) {
        const float m = __ldg(mask + p);
        if (m == 0.f) continue;
        const int y = p / W, x = p - y * W;
        float v = 0.f;
#pragma unroll
        for (int l = 0; l < LP_TAPS; ++l) {
            int y0, y1, x0, x1;
            float ly1, lx1;
            lp_bilinear_axis(sp.sy[l], y, sp.h[l], &y0, &y1, &ly1);
            lp_bilinear_axis(sp.sx[l], x, sp.w[l], &x0, &x1, &lx1);
            const float ly0 = 1.f - ly1, lx0 = 1.f - lx1;
            const float* r0 = sp.map[l] + (int64_t)y0 * sp.w[l];
            const float* r1 = sp.map[l] + (int64_t)y1 * sp.w[l];
            v += ly0 * (lx0 * __ldg(r0 + x0) + lx1 * __ldg(r0 + x1)) + ly1 * (lx0 * __ldg(r1 + x0) + lx1 * __ldg(r1 + x1));
        }
        am += (double)m * (double)v;
        an += (double)m;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        am += __shfl_xor_sync(0xffffffffu, am, o);
        an += __shfl_xor_sync(0xffffffffu, an, o);
    }
    if (lane == 0) {
        red[0][warp] = am;
        red[1][warp] = an;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, n = 0.0;
        for (int w = 0; w < LP_SPATIAL_THREADS / 32; ++w) {
            a += red[0][w];
            n += red[1][w];
        }
        part[blockIdx.x] = a;
        part[gridDim.x + blockIdx.x] = n;
    }
}

// part [2][ctas] -> out = (sum of part[0]) / (sum of part[1]), each summed in a fixed order; an empty mask gives 0 / 0 = NaN
__global__ void __launch_bounds__(256) lpips_masked_finalize_kernel(const double* __restrict__ part, int ctas,
                                                                    float* __restrict__ out) {
    __shared__ double sh[2][256];
    double a = 0.0, n = 0.0;
    for (int i = threadIdx.x; i < ctas; i += 256) {
        a += part[i];
        n += part[ctas + i];
    }
    sh[0][threadIdx.x] = a;
    sh[1][threadIdx.x] = n;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            sh[0][threadIdx.x] += sh[0][threadIdx.x + s];
            sh[1][threadIdx.x] += sh[1][threadIdx.x + s];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = (float)(sh[0][0] / sh[1][0]);
}

// ---- host entry points -------------------------------------------------------------------------------------------------

extern "C" int64_t rdg_lpips_packed_floats(int32_t net) {
    LpNet N;
    if (!lp_net(net, &N)) { rdg_set_error("%s: unknown net %d (RDG_LPIPS_ALEX or RDG_LPIPS_VGG)", __func__, net); return RDG_E_ARG; }
    LpPacked P;
    lp_packed_layout(N, &P);
    return P.total;
}

extern "C" int rdg_lpips_pack(int32_t net, const float* const* conv_w, const float* const* conv_b, const float* const* lin_w,
                              float* packed, int64_t packed_floats, void* stream) {
    LpNet N;
    if (!lp_net(net, &N)) { rdg_set_error("%s: unknown net %d (RDG_LPIPS_ALEX or RDG_LPIPS_VGG)", __func__, net); return RDG_E_ARG; }
    RDG_CHECK_ARG(conv_w, "conv_w is NULL");
    RDG_CHECK_ARG(conv_b, "conv_b is NULL");
    RDG_CHECK_ARG(lin_w, "lin_w is NULL");
    RDG_CHECK_ARG(packed, "packed is NULL");
    LpPacked P;
    lp_packed_layout(N, &P);
    RDG_CHECK_ARG(packed_floats == P.total, "packed_floats is not rdg_lpips_packed_floats(net)");
    RDG_CHECK_ARG(((uintptr_t)packed & 15) == 0, "packed must be 16-byte aligned");
    int nconv = 0, ntap = 0;
    for (int i = 0; i < N.n; ++i) {
        if (!N.layers[i].conv) continue;
        if (!conv_w[nconv]) { rdg_set_error("%s: conv_w[%d] is NULL", __func__, nconv); return RDG_E_ARG; }
        if (!conv_b[nconv]) { rdg_set_error("%s: conv_b[%d] is NULL", __func__, nconv); return RDG_E_ARG; }
        if (N.layers[i].tap && !lin_w[ntap]) { rdg_set_error("%s: lin_w[%d] is NULL", __func__, ntap); return RDG_E_ARG; }
        ntap += N.layers[i].tap;
        ++nconv;
    }
    cudaStream_t s = (cudaStream_t)stream;
    int launches = 0;
    nconv = ntap = 0;
    for (int i = 0; i < N.n; ++i) {
        const LpLayer& L = N.layers[i];
        if (!L.conv) continue;
        const int kpad = lp_kpad(L);
        const int64_t n = (int64_t)L.cout * kpad;
        lpips_pack_kernel<<<(unsigned)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096), 256, 0, s>>>(
            conv_w[nconv], packed + P.w_off[i], L.cin, L.cout, L.k, kpad, lp_bn(L.cout));
        RDG_CHECK_LAUNCH();
        lpips_copy_kernel<<<rdg_div_up(L.cout, 256), 256, 0, s>>>(conv_b[nconv], packed + P.b_off[i], L.cout);
        RDG_CHECK_LAUNCH();
        launches += 2;
        if (L.tap) {
            lpips_copy_kernel<<<rdg_div_up(L.cout, 256), 256, 0, s>>>(lin_w[ntap], packed + P.lin_off[ntap], L.cout);
            RDG_CHECK_LAUNCH();
            ++launches;
            ++ntap;
        }
        ++nconv;
    }
    rdg_count_launches(launches);
    return RDG_OK;
}

static int lp_check_size(const char* fn, const LpNet& N, int32_t height, int32_t width) {
    if (height < N.min_edge) { rdg_set_error("%s: height must be >= %d for this net (got %d)", fn, N.min_edge, height); return RDG_E_ARG; }
    if (width < N.min_edge) { rdg_set_error("%s: width must be >= %d for this net (got %d)", fn, N.min_edge, width); return RDG_E_ARG; }
    // the conv tile's row index and the activation tensors of the pair stay within int32 / the grid
    if ((int64_t)height * width > (int64_t)1 << 26) { rdg_set_error("%s: height * width exceeds 2^26", fn); return RDG_E_ARG; }
    return RDG_OK;
}

static int64_t lp_workspace_bytes(const char* fn, int32_t net, int32_t height, int32_t width, bool masked) {
    LpNet N;
    if (!lp_net(net, &N)) { rdg_set_error("%s: unknown net %d (RDG_LPIPS_ALEX or RDG_LPIPS_VGG)", fn, net); return RDG_E_ARG; }
    const int rc = lp_check_size(fn, N, height, width);
    if (rc != RDG_OK) return rc;
    LpWork Wk;
    lp_work_layout(N, height, width, masked, &Wk);
    return Wk.total;
}

extern "C" int64_t rdg_lpips_workspace_bytes(int32_t net, int32_t height, int32_t width) {
    return lp_workspace_bytes(__func__, net, height, width, false);
}

extern "C" int64_t rdg_masked_lpips_workspace_bytes(int32_t net, int32_t height, int32_t width) {
    return lp_workspace_bytes(__func__, net, height, width, true);
}

#define LP_ARG(cond, msg)                                          \
    do {                                                           \
        if (!(cond)) {                                             \
            rdg_set_error("%s: %s", fn, msg);                      \
            return RDG_E_ARG;                                      \
        }                                                          \
    } while (0)

#define LP_LAUNCHED()                                                                   \
    do {                                                                                \
        cudaError_t e__ = cudaGetLastError();                                           \
        if (e__ != cudaSuccess) {                                                       \
            rdg_set_error("%s: CUDA error: %s", fn, cudaGetErrorString(e__));           \
            return RDG_E_CUDA;                                                          \
        }                                                                               \
    } while (0)

// rdg_lpips (mask == NULL) and rdg_masked_lpips: checks every argument, then runs the pairs in turn
static int lp_score(const char* fn, bool masked, const float* pred, const float* gt, const float* mask, int32_t batch,
                    int32_t channels, int32_t height, int32_t width, float value_range, int32_t net, const float* packed,
                    int64_t packed_floats, float* out, void* workspace, int64_t workspace_bytes, void* stream) {
    LP_ARG(pred, "pred is NULL");
    LP_ARG(gt, "gt is NULL");
    if (masked) LP_ARG(mask, "mask is NULL");
    LP_ARG(packed, "packed is NULL");
    LP_ARG(out, "out is NULL");
    LP_ARG(workspace, "workspace is NULL");
    LpNet N;
    if (!lp_net(net, &N)) { rdg_set_error("%s: unknown net %d (RDG_LPIPS_ALEX or RDG_LPIPS_VGG)", fn, net); return RDG_E_ARG; }
    LP_ARG(batch >= 1, "batch must be >= 1");
    LP_ARG(channels == 3, "channels must be 3 (LPIPS takes RGB images)");
    const int rc = lp_check_size(fn, N, height, width);
    if (rc != RDG_OK) return rc;
    LP_ARG(value_range > 0.0f && isfinite(value_range), "value_range must be a finite value > 0");
    LpPacked P;
    lp_packed_layout(N, &P);
    LP_ARG(packed_floats == P.total, "packed_floats is not rdg_lpips_packed_floats(net)");
    LP_ARG(((uintptr_t)packed & 15) == 0, "packed must be 16-byte aligned");
    LpWork Wk;
    lp_work_layout(N, height, width, masked, &Wk);
    LP_ARG(workspace_bytes >= Wk.total, masked ? "workspace_bytes is smaller than rdg_masked_lpips_workspace_bytes()"
                                               : "workspace_bytes is smaller than rdg_lpips_workspace_bytes()");
    LP_ARG(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");

    cudaStream_t s = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    float* act[2] = {(float*)ws, (float*)(ws + Wk.act_bytes)};
    {
        const cudaError_t e = cudaFuncSetAttribute(lpips_conv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kConvSmem);
        if (e != cudaSuccess) {
            rdg_set_error("%s: cudaFuncSetAttribute(lpips_conv_kernel) failed: %s", fn, cudaGetErrorString(e));
            return RDG_E_CUDA;
        }
    }
    LpFinal fin = {};
    LpSpatial sp = {};
    for (int l = 0; l < LP_TAPS; ++l) {
        if (masked) {
            sp.map[l] = (const float*)(ws + Wk.map_off[l]);
            sp.h[l] = Wk.tap_h[l];
            sp.w[l] = Wk.tap_w[l];
            sp.sy[l] = (float)Wk.tap_h[l] / (float)height;
            sp.sx[l] = (float)Wk.tap_w[l] / (float)width;
        } else {
            fin.part[l] = (const double*)(ws + Wk.part_off[l]);
            fin.ctas[l] = Wk.head_ctas[l];
            fin.positions[l] = (double)Wk.tap_h[l] * Wk.tap_w[l];
        }
    }
    double* spatial_part = masked ? (double*)(ws + Wk.spatial_off) : nullptr;
    const int64_t hw = (int64_t)height * width;
    int launches = 0;
    for (int b = 0; b < batch; ++b) {
        lpips_scale_kernel<<<(unsigned)((2 * hw + 255) / 256), 256, 0, s>>>(pred + b * 3 * hw, gt + b * 3 * hw,
                                                                              masked ? mask + b * hw : nullptr, height, width,
                                                                              value_range, act[0]);
        LP_LAUNCHED();
        ++launches;
        int cur = 0, h = height, w = width, t = 0;
        for (int i = 0; i < N.n; ++i) {
            const LpLayer& L = N.layers[i];
            const int ho = (h + 2 * L.p - L.k) / L.s + 1, wo = (w + 2 * L.p - L.k) / L.s + 1;
            if (L.conv) {
                LpConv c;
                c.in = act[cur];
                c.out = act[cur ^ 1];
                c.wpk = packed + P.w_off[i];
                c.bias = packed + P.b_off[i];
                c.H = h; c.W = w; c.cin = L.cin; c.Ho = ho; c.Wo = wo; c.cout = L.cout;
                c.k = L.k; c.s = L.s; c.p = L.p;
                c.M = 2 * ho * wo;
                c.kchunks = lp_kpad(L) / LP_BK;
                c.bn = lp_bn(L.cout);
                c.ntiles = L.cout / c.bn;
                const int64_t ctas = (int64_t)rdg_div_up(c.M, LP_BM) * c.ntiles;
                lpips_conv_kernel<<<(unsigned)ctas, LP_THREADS, kConvSmem, s>>>(c);
                LP_LAUNCHED();
                ++launches;
                if (L.tap) {
                    if (masked)
                        lpips_head_kernel<true><<<Wk.head_ctas[t], LP_HEAD_THREADS, 0, s>>>(
                            act[cur ^ 1], packed + P.lin_off[t], (int64_t)ho * wo, L.cout, nullptr, (float*)sp.map[t]);
                    else
                        lpips_head_kernel<false><<<Wk.head_ctas[t], LP_HEAD_THREADS, 0, s>>>(
                            act[cur ^ 1], packed + P.lin_off[t], (int64_t)ho * wo, L.cout, (double*)fin.part[t], nullptr);
                    LP_LAUNCHED();
                    ++launches;
                    ++t;
                }
            } else {
                const int64_t n = 2LL * ho * wo * (L.cin / 4);
                lpips_pool_kernel<<<(unsigned)((n + 255) / 256 < 8192 ? (n + 255) / 256 : 8192), 256, 0, s>>>(
                    (const float4*)act[cur], (float4*)act[cur ^ 1], h, w, L.cin / 4, ho, wo, L.k, L.s);
                LP_LAUNCHED();
                ++launches;
            }
            cur ^= 1;
            h = ho;
            w = wo;
        }
        if (masked) {
            lpips_spatial_kernel<<<Wk.spatial_ctas, LP_SPATIAL_THREADS, 0, s>>>(sp, mask + b * hw, height, width, spatial_part);
            LP_LAUNCHED();
            lpips_masked_finalize_kernel<<<1, 256, 0, s>>>(spatial_part, Wk.spatial_ctas, out + b);
            LP_LAUNCHED();
            launches += 2;
        } else {
            lpips_finalize_kernel<<<1, 256, 0, s>>>(fin, out + b);
            LP_LAUNCHED();
            ++launches;
        }
    }
    rdg_count_launches(launches);
    return RDG_OK;
}

extern "C" int rdg_lpips(const float* pred, const float* gt, int32_t batch, int32_t channels, int32_t height, int32_t width,
                         float value_range, int32_t net, const float* packed, int64_t packed_floats, float* out, void* workspace,
                         int64_t workspace_bytes, void* stream) {
    return lp_score(__func__, false, pred, gt, nullptr, batch, channels, height, width, value_range, net, packed, packed_floats,
                    out, workspace, workspace_bytes, stream);
}

extern "C" int rdg_masked_lpips(const float* pred, const float* gt, const float* mask, int32_t batch, int32_t channels,
                                int32_t height, int32_t width, float value_range, int32_t net, const float* packed,
                                int64_t packed_floats, float* out, void* workspace, int64_t workspace_bytes, void* stream) {
    return lp_score(__func__, true, pred, gt, mask, batch, channels, height, width, value_range, net, packed, packed_floats, out,
                    workspace, workspace_bytes, stream);
}
