// Exact K nearest neighbours of every point among the same n points - the search behind RigidityLoss
// (/root/reference/src/trainer/losses.py:238-239: `torch3d.knn_points(target_points[None], target_points[None], K)`,
// pytorch3d un-vendored; its CUDA kernel is an exhaustive O(n^2) scan, 2.5e11 distance evaluations for the
// 500 K sampled Gaussians of BASELINE config 4).
//
// B200 mapping: a uniform grid over the bounding box with ~2 points per cell, built on the device with no host
// round trip (bounding box -> cell size -> per-cell counts -> exclusive scan -> counting sort of (x, y, z, index)
// float4 records).  One thread per query walks the cube shells around its own cell; cells that are adjacent in x are
// adjacent in memory, so every shell row is ONE contiguous run of 16-byte records, and the queries of a warp are
// neighbours in space (they are processed in sorted order), so they read the same runs out of L1/L2.  The K best
// (distance, index) pairs stay in registers.  The walk stops after shell r once the K-th distance is strictly below
// (r * cell)^2 - everything unvisited is at least that far - which makes the result exact, not approximate.
//   Contract (the oracle's, oracle/motion_oracle.py::knn_points): squared distance (dx*dx + dy*dy) + dz*dz with one
//   float32 rounding per operation (explicit _rn intrinsics, no FMA contraction), K smallest ascending, the query
//   itself included, exact ties towards the lower index.  Indices are therefore bit-exact against the oracle.
// Bound: L2 / LSU latency (gathered 16-byte records), ~27 cells x 2 records per query; HBM traffic is 16 B x n x 3.
// The same grid build and walk also give simple-knn's distCUDA2 (rdg_knn3_mean_dist2) and the gradient of the distances
// for the pytorch3d.ops.knn_points drop-in (rdg_knn_dist2_bwd).
#include <float.h>
#include <math.h>
#include "common.cuh"

#define KNN_TARGET_OCC 2.0f
#define KNN_SCAN_THREADS 1024

struct KnnGrid {
    float ox, oy, oz;      // bounding-box minimum
    float cell, inv_cell;
    int gx, gy, gz;
    int ncell;
};

__device__ __forceinline__ uint32_t f2ord(float f) {
    const uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

__global__ void knn_init_kernel(uint32_t* __restrict__ bbox) {
    if (threadIdx.x < 3) bbox[threadIdx.x] = 0xffffffffu;        // minima
    else if (threadIdx.x < 6) bbox[threadIdx.x] = 0u;            // maxima
}

__global__ void __launch_bounds__(RDG_BLOCK) knn_bbox_kernel(int64_t n, const float* __restrict__ pts,
                                                             uint32_t* __restrict__ bbox) {
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int64_t i = (int64_t)blockIdx.x * RDG_BLOCK + threadIdx.x; i < n; i += (int64_t)gridDim.x * RDG_BLOCK) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            const float v = pts[i * 3 + d];
            lo[d] = fminf(lo[d], v);
            hi[d] = fmaxf(hi[d], v);
        }
    }
#pragma unroll
    for (int d = 0; d < 3; ++d) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[d] = fminf(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o));
            hi[d] = fmaxf(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(bbox + d, f2ord(lo[d]));
            atomicMax(bbox + 3 + d, f2ord(hi[d]));
        }
    }
}

// one thread: choose the cell size so that the grid has about n / KNN_TARGET_OCC cells and fits `cell_cap`
__global__ void knn_grid_kernel(int64_t n, const uint32_t* __restrict__ bbox, int cell_cap, KnnGrid* __restrict__ grid) {
    float lo[3], ext[3];
    float emax = 0.f;
    for (int d = 0; d < 3; ++d) {
        lo[d] = ord2f(bbox[d]);
        ext[d] = ord2f(bbox[3 + d]) - lo[d];
        emax = fmaxf(emax, ext[d]);
    }
    if (!(emax > 0.f)) emax = 1.f;                       // all points identical
    // degenerate (flat) directions count as one thin slab
    float vol = 1.f;
    for (int d = 0; d < 3; ++d) vol *= fmaxf(ext[d], emax * 1e-3f);
    float cell = cbrtf(vol * KNN_TARGET_OCC / (float)n);
    cell = fmaxf(cell, emax * (1.0f / 1000.0f));          // at most ~1000 cells along an axis
    int g[3];
    for (int it = 0; it < 64; ++it) {
        int64_t total = 1;
        for (int d = 0; d < 3; ++d) {
            g[d] = (int)floorf(ext[d] / cell) + 1;
            total *= g[d];
        }
        if (total <= (int64_t)cell_cap) break;
        cell *= 1.26f;
    }
    grid->ox = lo[0]; grid->oy = lo[1]; grid->oz = lo[2];
    grid->cell = cell;
    grid->inv_cell = 1.0f / cell;
    grid->gx = g[0]; grid->gy = g[1]; grid->gz = g[2];
    grid->ncell = g[0] * g[1] * g[2];
}

__device__ __forceinline__ void cell_of(const KnnGrid& g, float x, float y, float z, int& cx, int& cy, int& cz) {
    cx = min(max((int)floorf((x - g.ox) * g.inv_cell), 0), g.gx - 1);
    cy = min(max((int)floorf((y - g.oy) * g.inv_cell), 0), g.gy - 1);
    cz = min(max((int)floorf((z - g.oz) * g.inv_cell), 0), g.gz - 1);
}

__global__ void __launch_bounds__(RDG_BLOCK) knn_count_kernel(int64_t n, const float* __restrict__ pts,
                                                              const KnnGrid* __restrict__ grid, uint32_t* __restrict__ count,
                                                              uint32_t* __restrict__ cell_id) {
    const KnnGrid g = *grid;
    for (int64_t i = (int64_t)blockIdx.x * RDG_BLOCK + threadIdx.x; i < n; i += (int64_t)gridDim.x * RDG_BLOCK) {
        int cx, cy, cz;
        cell_of(g, pts[i * 3], pts[i * 3 + 1], pts[i * 3 + 2], cx, cy, cz);
        const uint32_t c = (uint32_t)((cz * g.gy + cy) * g.gx + cx);
        cell_id[i] = c;
        atomicAdd(count + c, 1u);
    }
}

// exclusive scan of count[0 .. m) into start[0 .. m], one CTA (m <= a few million: two passes over an L2-resident array)
__global__ void __launch_bounds__(KNN_SCAN_THREADS) knn_scan_kernel(const uint32_t* __restrict__ count, int m,
                                                                     uint32_t* __restrict__ start) {
    __shared__ uint32_t warp_tot[KNN_SCAN_THREADS / 32];
    const int per = (m + KNN_SCAN_THREADS - 1) / KNN_SCAN_THREADS;
    const int b = threadIdx.x * per, e = min(b + per, m);
    uint32_t s = 0;
    for (int i = b; i < e; ++i) s += count[i];
    // block-wide exclusive scan of the per-thread sums
    uint32_t inc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
        if ((threadIdx.x & 31) >= o) inc += v;
    }
    if ((threadIdx.x & 31) == 31) warp_tot[threadIdx.x >> 5] = inc;
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t w = warp_tot[threadIdx.x];
        uint32_t winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, winc, o);
            if (threadIdx.x >= o) winc += v;
        }
        warp_tot[threadIdx.x] = winc - w;
    }
    __syncthreads();
    uint32_t run = warp_tot[threadIdx.x >> 5] + inc - s;
    for (int i = b; i < e; ++i) {
        start[i] = run;
        run += count[i];
    }
    if (threadIdx.x == KNN_SCAN_THREADS - 1) start[m] = run;   // the last thread's range ends at m (possibly empty)
}

__global__ void __launch_bounds__(RDG_BLOCK) knn_fill_kernel(int64_t n, const float* __restrict__ pts,
                                                             const uint32_t* __restrict__ cell_id,
                                                             const uint32_t* __restrict__ start, uint32_t* __restrict__ count,
                                                             float4* __restrict__ sorted) {
    for (int64_t i = (int64_t)blockIdx.x * RDG_BLOCK + threadIdx.x; i < n; i += (int64_t)gridDim.x * RDG_BLOCK) {
        const uint32_t c = cell_id[i];
        const uint32_t slot = start[c] + atomicSub(count + c, 1u) - 1u;   // the order inside a cell does not matter
        sorted[slot] = make_float4(pts[i * 3], pts[i * 3 + 1], pts[i * 3 + 2], __int_as_float((int)i));
    }
}

__device__ __forceinline__ bool pair_less(float da, int ia, float db, int ib) { return da < db || (da == db && ia < ib); }

// MEAN3 is simple-knn's distCUDA2: K = 3, the query itself is skipped BY INDEX (an exact duplicate is another point at
// distance 0 and may sort ahead of it), and the output is one float per point, ((b0 + b1) + b2) / 3 with b ascending.
template <int KMAX, bool MEAN3>
__global__ void __launch_bounds__(128) knn_query_kernel(int64_t n, int K, const float4* __restrict__ sorted,
                                                        const uint32_t* __restrict__ start, const KnnGrid* __restrict__ grid,
                                                        int32_t* __restrict__ out_idx, float* __restrict__ out_d) {
    const int64_t s = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (s >= n) return;
    const KnnGrid g = *grid;
    const float4 q = sorted[s];
    const int qi = __float_as_int(q.w);
    int cx, cy, cz;
    cell_of(g, q.x, q.y, q.z, cx, cy, cz);
    float bd[KMAX];
    int bi[KMAX];
#pragma unroll
    for (int j = 0; j < KMAX; ++j) { bd[j] = FLT_MAX; bi[j] = 0x7fffffff; }
    const int rmax = max(g.gx, max(g.gy, g.gz));
    for (int r = 0; r <= rmax; ++r) {
        const int z0 = max(cz - r, 0), z1 = min(cz + r, g.gz - 1);
        const int y0 = max(cy - r, 0), y1 = min(cy + r, g.gy - 1);
        for (int z = z0; z <= z1; ++z) {
            const bool zface = (z == cz - r) || (z == cz + r);
            for (int y = y0; y <= y1; ++y) {
                const bool face = zface || (y == cy - r) || (y == cy + r);
                // a face row spans the whole x range of the shell; an interior row only its two end cells
                const int nseg = (face || r == 0) ? 1 : 2;
                for (int seg = 0; seg < nseg; ++seg) {
                    int xa, xb;
                    if (nseg == 1) { xa = cx - r; xb = cx + r; }
                    else { xa = xb = seg ? cx + r : cx - r; }
                    if (xb < 0 || xa >= g.gx) continue;
                    xa = max(xa, 0);
                    xb = min(xb, g.gx - 1);
                    const int row = (z * g.gy + y) * g.gx;
                    const uint32_t pb = start[row + xa], pe = start[row + xb + 1];
                    for (uint32_t p = pb; p < pe; ++p) {
                        const float4 c = sorted[p];
                        const float dx = __fsub_rn(q.x, c.x), dy = __fsub_rn(q.y, c.y), dz = __fsub_rn(q.z, c.z);
                        const float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
                        const int ci = __float_as_int(c.w);
                        if (MEAN3 && ci == qi) continue;
                        bool worse = true;   // candidate vs the current K-th best
#pragma unroll
                        for (int j = 0; j < KMAX; ++j)
                            if (j == K - 1) worse = !pair_less(d, ci, bd[j], bi[j]);
                        if (worse) continue;
                        // insertion into the ascending list, every slot from the old values (descending j)
#pragma unroll
                        for (int j = KMAX - 1; j > 0; --j) {
                            if (j < K) {
                                const bool before_prev = pair_less(d, ci, bd[j - 1], bi[j - 1]);
                                const bool before_here = pair_less(d, ci, bd[j], bi[j]);
                                const float nd = before_prev ? bd[j - 1] : (before_here ? d : bd[j]);
                                const int ni = before_prev ? bi[j - 1] : (before_here ? ci : bi[j]);
                                bd[j] = nd; bi[j] = ni;
                            }
                        }
                        if (pair_less(d, ci, bd[0], bi[0])) { bd[0] = d; bi[0] = ci; }
                    }
                }
            }
        }
        // every unvisited point lies in a cell at Chebyshev distance >= r + 1, i.e. at least r * cell away
        float kth = FLT_MAX;
#pragma unroll
        for (int j = 0; j < KMAX; ++j)
            if (j == K - 1) kth = bd[j];
        const float bound = fmaxf((float)r - 0.01f, 0.f) * g.cell;   // 1 % slack for the rounding of the cell index
        if (kth < bound * bound) break;
    }
    if (MEAN3) {
        out_d[qi] = __fdiv_rn(__fadd_rn(__fadd_rn(bd[0], bd[1]), bd[2]), 3.0f);
        return;
    }
#pragma unroll
    for (int j = 0; j < KMAX; ++j)
        if (j < K) {
            out_idx[(int64_t)qi * K + j] = bi[j];
            out_d[(int64_t)qi * K + j] = bd[j];
        }
}

struct KnnLayout { int64_t bbox, grid, count, start, cell_id, sorted, total; int cell_cap; };

static KnnLayout knn_layout(int64_t n) {
    KnnLayout L;
    int64_t cap = n / 2 + 64;
    if (cap > (int64_t)1 << 26) cap = (int64_t)1 << 26;
    L.cell_cap = (int)cap;
    int64_t off = 0;
    L.bbox = off; off += 256;
    L.grid = off; off += 256;
    L.count = off; off += rdg_align_up((cap + 1) * 4, 256);
    L.start = off; off += rdg_align_up((cap + 2) * 4, 256);
    L.cell_id = off; off += rdg_align_up(n * 4, 256);
    L.sorted = off; off += rdg_align_up(n * 16, 256);
    L.total = off;
    return L;
}

extern "C" int64_t rdg_knn_workspace_bytes(int64_t n) { return n > 0 ? knn_layout(n).total : 0; }

// bounding box -> cell size -> per-cell counts -> exclusive scan -> counting sort; 6 launches, no host round trip
static int knn_build_grid(int64_t n, const float* points, const KnnLayout& L, char* ws, cudaStream_t st) {
    uint32_t* bbox = (uint32_t*)(ws + L.bbox);
    KnnGrid* grid = (KnnGrid*)(ws + L.grid);
    uint32_t* count = (uint32_t*)(ws + L.count);
    uint32_t* start = (uint32_t*)(ws + L.start);
    uint32_t* cell_id = (uint32_t*)(ws + L.cell_id);
    float4* sorted = (float4*)(ws + L.sorted);
    const int64_t want = (n + RDG_BLOCK - 1) / RDG_BLOCK;
    const int pgrid = (int)(want < (int64_t)RDG_SM_COUNT * 8 ? want : (int64_t)RDG_SM_COUNT * 8);
    knn_init_kernel<<<1, 32, 0, st>>>(bbox);
    RDG_CUDA(cudaMemsetAsync(count, 0, (size_t)(L.cell_cap + 1) * 4, st));
    knn_bbox_kernel<<<pgrid, RDG_BLOCK, 0, st>>>(n, points, bbox);
    knn_grid_kernel<<<1, 1, 0, st>>>(n, bbox, L.cell_cap, grid);
    knn_count_kernel<<<pgrid, RDG_BLOCK, 0, st>>>(n, points, grid, count, cell_id);
    knn_scan_kernel<<<1, KNN_SCAN_THREADS, 0, st>>>(count, L.cell_cap, start);
    knn_fill_kernel<<<pgrid, RDG_BLOCK, 0, st>>>(n, points, cell_id, start, count, sorted);
    return RDG_OK;
}

extern "C" int rdg_knn(int64_t n, const float* points, int32_t K, int32_t* idx, float* dist2, void* workspace,
                       int64_t workspace_bytes, void* stream) {
    RDG_CHECK_ARG(points && idx && dist2 && workspace, "null argument");
    RDG_CHECK_ARG(K >= 1 && K <= 16, "K must be in 1..16");
    RDG_CHECK_ARG(n >= K, "fewer points than neighbours requested");
    RDG_CHECK_ARG(n < ((int64_t)1 << 31), "too many points");
    const KnnLayout L = knn_layout(n);
    RDG_CHECK_ARG(workspace_bytes >= L.total, "workspace too small (rdg_knn_workspace_bytes)");
    RDG_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    const int rc = knn_build_grid(n, points, L, ws, st);
    if (rc != RDG_OK) return rc;
    const float4* sorted = (const float4*)(ws + L.sorted);
    const uint32_t* start = (const uint32_t*)(ws + L.start);
    const KnnGrid* grid = (const KnnGrid*)(ws + L.grid);
    const int qgrid = rdg_div_up(n, 128);
    if (K <= 8) knn_query_kernel<8, false><<<qgrid, 128, 0, st>>>(n, K, sorted, start, grid, idx, dist2);
    else knn_query_kernel<16, false><<<qgrid, 128, 0, st>>>(n, K, sorted, start, grid, idx, dist2);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(7);
    return RDG_OK;
}

extern "C" int rdg_knn3_mean_dist2(int64_t n, const float* points, float* out, void* workspace, int64_t workspace_bytes,
                                   void* stream) {
    RDG_CHECK_ARG(points && out && workspace, "null argument");
    RDG_CHECK_ARG(n >= 4, "distCUDA2 needs at least 4 points (3 neighbours besides the point itself)");
    RDG_CHECK_ARG(n < ((int64_t)1 << 31), "too many points");
    const KnnLayout L = knn_layout(n);
    RDG_CHECK_ARG(workspace_bytes >= L.total, "workspace too small (rdg_knn_workspace_bytes)");
    RDG_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    const int rc = knn_build_grid(n, points, L, ws, st);
    if (rc != RDG_OK) return rc;
    knn_query_kernel<3, true><<<rdg_div_up(n, 128), 128, 0, st>>>(
        n, 3, (const float4*)(ws + L.sorted), (const uint32_t*)(ws + L.start), (const KnnGrid*)(ws + L.grid), nullptr, out);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(7);
    return RDG_OK;
}

// dist2[i, k] = |p_i - p_j|^2 with j = idx[i, k]: d/dp_i = 2 g (p_i - p_j) summed over k in registers (every row is one
// thread's), d/dp_j = -2 g (p_i - p_j) scattered with float atomics (a point is the neighbour of many rows).
__global__ void __launch_bounds__(RDG_BLOCK) knn_dist2_bwd_kernel(int64_t n, int K, const float* __restrict__ pts,
                                                                  const int32_t* __restrict__ idx,
                                                                  const float* __restrict__ g,
                                                                  float* __restrict__ d_query, float* __restrict__ d_ref) {
    const int64_t i = (int64_t)blockIdx.x * RDG_BLOCK + threadIdx.x;
    if (i >= n) return;
    const float px = pts[i * 3], py = pts[i * 3 + 1], pz = pts[i * 3 + 2];
    float ax = 0.f, ay = 0.f, az = 0.f;
    for (int k = 0; k < K; ++k) {
        const int64_t j = idx[i * K + k];
        const float g2 = 2.0f * g[i * K + k];
        const float cx = g2 * (px - pts[j * 3]), cy = g2 * (py - pts[j * 3 + 1]), cz = g2 * (pz - pts[j * 3 + 2]);
        ax += cx; ay += cy; az += cz;
        if (d_ref) {
            atomicAdd(d_ref + j * 3, -cx);
            atomicAdd(d_ref + j * 3 + 1, -cy);
            atomicAdd(d_ref + j * 3 + 2, -cz);
        }
    }
    if (d_query) {
        d_query[i * 3] = ax;
        d_query[i * 3 + 1] = ay;
        d_query[i * 3 + 2] = az;
    }
}

extern "C" int rdg_knn_dist2_bwd(int64_t n, int32_t K, const float* points, const int32_t* idx, const float* d_dist2,
                                 float* d_query, float* d_ref, void* stream) {
    RDG_CHECK_ARG(points && idx && d_dist2, "null argument");
    RDG_CHECK_ARG(K >= 1 && K <= 16, "K must be in 1..16");
    RDG_CHECK_ARG(n >= K && n < ((int64_t)1 << 31), "n out of range");
    if (!d_query && !d_ref) return RDG_OK;
    knn_dist2_bwd_kernel<<<rdg_div_up(n, RDG_BLOCK), RDG_BLOCK, 0, (cudaStream_t)stream>>>(n, K, points, idx, d_dist2,
                                                                                          d_query, d_ref);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}
