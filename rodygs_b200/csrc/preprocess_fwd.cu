// Fused per-Gaussian forward: static||dynamic fetch -> activations -> time-conditioned
// deformation -> EWA projection -> conic/radius/tile rectangle -> SH->RGB.
// SURVEY.md §8 rows a2-a7; spec: SURVEY.md App. A.2 == oracle/splat_oracle.py::preprocess.
//
// THIS TRANSLATION UNIT IS COMPILED WITH -fmad=false: depth bits, pixel centre,
// radius and tile rectangle must be bit-identical to the oracle's individually
// rounded float32 operations.  The kernel is HBM-bound, so the lost FMA contraction
// costs nothing.
//
// Roofline: HBM.  Algorithmic bytes per Gaussian (degree 3): read 44 (xyz, scale,
// quat, opacity) + 192 (SH) [+ 68 dynamic: coeff + birth index], write 8 (radii,
// tiles_touched) + 41 for visible ones (p0, p1, p2, clamped).
//
// B200 mapping: one thread per Gaussian, 256-Gaussian chunks that never straddle the
// static/dynamic boundary, so a chunk's higher-order SH rows are one contiguous,
// 16-byte aligned 46 KB span: it is fetched by ONE cp.async.bulk (TMA) into shared memory
// while the threads load their 44 B of geometry and run the projection; each thread then
// reads its own row (stride 45 words: conflict-free).  46 KB per CTA -> 4 CTAs per SM.
#include "scene.cuh"
#include "tma.cuh"

#define SH_ROW 45  // odd row stride in shared memory: conflict-free per-thread row reads

struct PreFwdParams {
    RdgScene sc;
    RdgView view;
    RdgGeom geom;
    int use_tma;
    int diff_smem;   // B(t) - table rows staged in shared memory (rdg_stage_diff); the launcher sized the buffer
    int l2_prefetch; // next chunk's parameter rows prefetched into L2 (cp.async.bulk.prefetch.L2)
};

// ---- the per-view arithmetic, shared by preprocess_fwd_kernel and the batched preprocess_fwd_views_kernel ----

// A Gaussian's screen-space footprint in one view.  Zero / false = culled.
struct RdgFootprint {
    float px = 0.f, py = 0.f, conA = 0.f, conB = 0.f, conC = 0.f, tz = 0.f;
    int radius = 0;
    unsigned tiles = 0;
    bool vis = false;
};

// EWA projection -> conic, radius, pixel centre and tile rectangle of the activated (deformed) Gaussian a, and its
// per-tile population count (geom.tile_count, when set).  Writes geom.dbg_activated[i] when set.
__device__ __forceinline__ void rdg_fwd_footprint(const RdgGeom& geom, int64_t i, const RdgCam& cam, const RdgAct& a,
                                                  float scale_modifier, RdgFootprint& f) {
    if (geom.dbg_activated) {
        float* d = geom.dbg_activated + i * 11;
        d[0] = a.x; d[1] = a.y; d[2] = a.z; d[3] = a.s[0]; d[4] = a.s[1]; d[5] = a.s[2];
        d[6] = a.q[0]; d[7] = a.q[1]; d[8] = a.q[2]; d[9] = a.q[3]; d[10] = a.op;
    }
    RdgProj pr;
    rdg_project(cam, a, scale_modifier, pr);
    if (pr.tz > RDG_NEAR_Z && pr.det != 0.0f) {
        const float det_inv = 1.0f / pr.det;
        f.conA = pr.cc * det_inv; f.conB = -pr.cb * det_inv; f.conC = pr.ca * det_inv;
        const float mid = 0.5f * (pr.ca + pr.cc);
        const float disc = sqrtf(fmaxf(0.1f, mid * mid - pr.det));
        const float lam1 = mid + disc, lam2 = mid - disc;
        const float rad_f = ceilf(3.0f * sqrtf(fmaxf(lam1, lam2)));
        const float ndcx = pr.hx * pr.pw, ndcy = pr.hy * pr.pw;
        f.px = ((ndcx + 1.0f) * cam.W - 1.0f) * 0.5f;
        f.py = ((ndcy + 1.0f) * cam.H - 1.0f) * 0.5f;
        const int rminx = min(cam.gx, max(0, (int)((f.px - rad_f) / 16.0f)));
        const int rminy = min(cam.gy, max(0, (int)((f.py - rad_f) / 16.0f)));
        const int rmaxx = min(cam.gx, max(0, (int)((f.px + rad_f + 15.0f) / 16.0f)));
        const int rmaxy = min(cam.gy, max(0, (int)((f.py + rad_f + 15.0f) / 16.0f)));
        const int cntt = (rmaxx - rminx) * (rmaxy - rminy);
        if (cntt > 0) {
            f.radius = (int)rad_f; f.tiles = (unsigned)cntt; f.vis = true; f.tz = pr.tz;
            if (geom.tile_count) {   // per-tile population for the tile-bucketed binning
                for (int yy = rminy; yy < rmaxy; ++yy)
                    for (int xx = rminx; xx < rmaxx; ++xx) atomicAdd(&geom.tile_count[yy * cam.gx + xx], 1u);
            }
        }
    }
}

// SH -> RGB for the camera at campos (rest: the Gaussian's higher-order SH row in shared memory) and the stores of row i.
template <int DEG>
__device__ __forceinline__ void rdg_fwd_finish(const RdgGeom& geom, const RdgScene& sc, int64_t i, bool valid,
                                               const RdgFootprint& f, const RdgAct& a, const float* campos, float dc0,
                                               float dc1, float dc2, const float* rest) {
    constexpr int K = (DEG + 1) * (DEG + 1);
    if (f.vis) {
        float rgb[3];
        unsigned clamped = 0;
        if (sc.colors_precomp) {
            rgb[0] = sc.colors_precomp[i * 3 + 0];
            rgb[1] = sc.colors_precomp[i * 3 + 1];
            rgb[2] = sc.colors_precomp[i * 3 + 2];
        } else {
            float dx = a.x - campos[0], dy = a.y - campos[1], dz = a.z - campos[2];
            const float inv = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz);
            dx *= inv; dy *= inv; dz *= inv;
            float b[K];
            rdg_sh_basis<DEG>(dx, dy, dz, b);
            rgb[0] = b[0] * dc0; rgb[1] = b[0] * dc1; rgb[2] = b[0] * dc2;
#pragma unroll
            for (int k = 1; k < K; ++k) {   // explicit FMAs (-fmad=false TU): the colour feeds no integer output
                rgb[0] = fmaf(b[k], rest[(k - 1) * 3 + 0], rgb[0]);
                rgb[1] = fmaf(b[k], rest[(k - 1) * 3 + 1], rgb[1]);
                rgb[2] = fmaf(b[k], rest[(k - 1) * 3 + 2], rgb[2]);
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                rgb[c] += 0.5f;
                if (rgb[c] < 0.0f) { clamped |= 1u << c; rgb[c] = 0.0f; }
            }
        }
        reinterpret_cast<float4*>(geom.p0)[i] = make_float4(f.px, f.py, f.conA, f.conB);
        reinterpret_cast<float4*>(geom.p1)[i] = make_float4(f.conC, a.op, rgb[0], rgb[1]);
        reinterpret_cast<float2*>(geom.p2)[i] = make_float2(rgb[2], f.tz);
        geom.clamped[i] = (uint8_t)clamped;
    }
    if (valid) {
        geom.radii[i] = f.radius;
        geom.tiles_touched[i] = f.tiles;
    }
}

// Measured alternatives that did NOT help (B200, C4, profiles/r01_ab_v12_*.json, r01_ab_v13_*.json): double-buffering the SH
// rows (next chunk's bulk load issued one chunk ahead; 0.266 vs 0.258 ms - the bulk copy is not what the warps wait for)
// and forcing 3 CTAs per SM with __launch_bounds__(256, 3) (80 registers + spills; 0.302 vs 0.259 ms).
template <bool RAW, int DEG>
__global__ void __launch_bounds__(RDG_BLOCK) preprocess_fwd_kernel(const PreFwdParams p) {
    extern __shared__ __align__(128) float smem[];
    constexpr int K = (DEG + 1) * (DEG + 1);
    constexpr int NREST = 3 * (K - 1);
    const RdgScene& sc = p.sc;
    float* sh_s = smem;                       // [256][SH_ROW]
    float* bt_s = smem + RDG_BLOCK * SH_ROW;  // [16*7] B(t)
    __shared__ __align__(8) uint64_t bar;

    RdgCam cam;
    rdg_load_cam(cam, p.view.viewmatrix, p.view.projmatrix, p.view.tanfovx, p.view.tanfovy,
                 p.view.width, p.view.height);
    float campos[3];
    rdg_campos(cam, campos);

    const bool deform = RAW && sc.use_deform && sc.n_dynamic > 0;
    float* diff_s = (deform && p.diff_smem) ? bt_s + RDG_NUM_BASIS_MAX * 7 : nullptr;
    if (deform) {
        for (int e = threadIdx.x; e < sc.num_basis * 7; e += RDG_BLOCK) bt_s[e] = sc.basis_t[e];
        if (diff_s) rdg_stage_diff(sc, sc.basis_t, diff_s, RDG_BLOCK);
    }
    if (threadIdx.x == 0) rdg_mbar_init(&bar, 1);
    __syncthreads();

    const bool use_sh = (sc.colors_precomp == nullptr) && NREST > 0;
    const int64_t cs = (sc.n_static + RDG_BLOCK - 1) / RDG_BLOCK, cd = (sc.n_dynamic + RDG_BLOCK - 1) / RDG_BLOCK;
    uint32_t phase = 0;
    for (int64_t chunk = blockIdx.x; chunk < cs + cd; chunk += gridDim.x) {
        const bool dyn = chunk >= cs;
        const RdgSet& set = dyn ? sc.dy : sc.st;
        const int64_t lbase = (dyn ? chunk - cs : chunk) * RDG_BLOCK;
        const int64_t n_set = dyn ? sc.n_dynamic : sc.n_static;
        const int cnt = (int)min((int64_t)RDG_BLOCK, n_set - lbase);
        if (p.l2_prefetch && chunk + gridDim.x < cs + cd && threadIdx.x < 8)
            rdg_prefetch_chunk_field(sc, chunk + gridDim.x, cs, threadIdx.x, nullptr);

        // ---- stage this chunk's higher-order SH rows in shared memory ----
        bool tma = false;
        if (use_sh) {
            __syncthreads();  // previous chunk's readers are done with sh_s
            tma = p.use_tma && NREST == SH_ROW && set.sh_rest_stride == SH_ROW && (cnt & 3) == 0;
            if (tma) {
                if (threadIdx.x == 0) {
                    rdg_fence_proxy_async();
                    rdg_bulk_load(sh_s, set.sh_rest + lbase * SH_ROW, (uint32_t)(cnt * SH_ROW * sizeof(float)), &bar);
                }
            } else if (set.sh_rest_stride == NREST) {
                const float* src = set.sh_rest + lbase * NREST;
                for (int e = threadIdx.x; e < cnt * NREST; e += RDG_BLOCK) sh_s[(e / NREST) * SH_ROW + (e % NREST)] = src[e];
            } else {
                const int stride = set.sh_rest_stride;   // e.g. 48: cat'ed [n,16,3] rows of the drop-in boundary
                const float* src = set.sh_rest + lbase * stride;
                for (int e = threadIdx.x; e < cnt * NREST; e += RDG_BLOCK) {
                    const int g = e / NREST, k = e - g * NREST;
                    sh_s[g * SH_ROW + k] = src[(int64_t)g * stride + k];
                }
            }
        }

        const bool valid = (int)threadIdx.x < cnt;
        const int64_t local = lbase + threadIdx.x;
        const int64_t i = (dyn ? sc.n_static : 0) + local;
        RdgFootprint f;
        RdgAct a;
        // degree-0 SH coefficients: requested here with the geometry, not after the SH rows have arrived - otherwise they
        // are one more exposed DRAM round trip at the end of every chunk (the kernel is latency bound)
        float dc0 = 0.f, dc1 = 0.f, dc2 = 0.f;
        if (valid && !sc.colors_precomp) {
            const float* dc = set.sh_dc + local * set.sh_dc_stride;
            dc0 = __ldg(dc); dc1 = __ldg(dc + 1); dc2 = __ldg(dc + 2);
        }
        if (valid) {
            rdg_fetch<RAW>(sc, dyn, local, bt_s, a, diff_s);
            rdg_fwd_footprint(p.geom, i, cam, a, p.view.scale_modifier, f);
        }
        if (use_sh) {
            if (tma) rdg_mbar_wait(&bar, phase & 1u);
            else __syncthreads();
        }
        if (tma) ++phase;
        rdg_fwd_finish<DEG>(p.geom, sc, i, valid, f, a, campos, dc0, dc1, dc2, sh_s + threadIdx.x * SH_ROW);
    }
}

template <bool RAW, int DEG>
static int launch_fwd(const PreFwdParams& p, int grid, size_t smem, cudaStream_t s) {
    const int cap = rdg_tunable(RDG_TUN_PRE_GRID_CAP);
    if (cap > 0 && grid > cap) grid = cap;
    RDG_CUDA(cudaFuncSetAttribute(preprocess_fwd_kernel<RAW, DEG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    preprocess_fwd_kernel<RAW, DEG><<<grid, RDG_BLOCK, smem, s>>>(p);
    RDG_CHECK_LAUNCH();
    return RDG_OK;
}

template <bool RAW>
static int launch_fwd_deg(const PreFwdParams& p, int deg, int grid, size_t smem, cudaStream_t s) {
    switch (deg) {
        case 0: return launch_fwd<RAW, 0>(p, grid, smem, s);
        case 1: return launch_fwd<RAW, 1>(p, grid, smem, s);
        case 2: return launch_fwd<RAW, 2>(p, grid, smem, s);
        default: return launch_fwd<RAW, 3>(p, grid, smem, s);
    }
}

// Argument checks shared by rdg_preprocess_fwd and rdg_preprocess_fwd_views: the message of the first failed check, or NULL.
static const char* view_arg_error(const RdgView* view) {
    if (!(view->sh_degree >= 0 && view->sh_degree <= 3)) return "sh_degree must be 0..3";
    if (!(view->width > 0 && view->height > 0)) return "empty image";
    if (!(view->viewmatrix && view->projmatrix)) return "null camera matrix";
    return nullptr;
}

static bool geom_complete(const RdgGeom* geom) {
    return geom->radii && geom->tiles_touched && geom->p0 && geom->p1 && geom->p2 && geom->clamped;
}

// basis_t: where B(t) comes from (scene->basis_t for one view, basis_ts for several)
static const char* scene_arg_error(const RdgScene* scene, int sh_degree, const float* basis_t) {
    if (!(scene->n_static == 0 || (scene->st.xyz && scene->st.scaling && scene->st.rotation && scene->st.opacity)))
        return "null static parameter";
    if (!(scene->n_dynamic == 0 || (scene->dy.xyz && scene->dy.scaling && scene->dy.rotation && scene->dy.opacity)))
        return "null dynamic parameter";
    if (!(scene->colors_precomp || ((scene->n_static == 0 || scene->st.sh_dc) && (scene->n_dynamic == 0 || scene->dy.sh_dc))))
        return "exactly one of SHs / precomputed colours is required";
    if (!(scene->colors_precomp || sh_degree == 0 ||
          ((scene->n_static == 0 || scene->st.sh_rest) && (scene->n_dynamic == 0 || scene->dy.sh_rest))))
        return "null higher-order SH pointer";
    if (scene->raw && scene->use_deform && scene->n_dynamic > 0) {
        if (!(scene->num_basis > 0 && scene->num_basis <= RDG_NUM_BASIS_MAX)) return "num_basis out of range";
        if (!(scene->motion_coeff && scene->time_ind && basis_t && scene->table && scene->num_times > 0))
            return "null deformation input";
    }
    return nullptr;
}

extern "C" int rdg_preprocess_fwd(const RdgScene* scene, const RdgView* view, const RdgGeom* geom, void* stream) {
    RDG_CHECK_ARG(scene && view && geom, "null argument");
    const int64_t N = scene->n_static + scene->n_dynamic;
    RDG_CHECK_ARG(N >= 0 && scene->n_static >= 0 && scene->n_dynamic >= 0, "negative count");
    const char* err = view_arg_error(view);
    RDG_CHECK_ARG(!err, err);
    if (N == 0) return RDG_OK;
    RDG_CHECK_ARG(geom_complete(geom), "null geometry buffer");
    err = scene_arg_error(scene, view->sh_degree, scene->basis_t);
    RDG_CHECK_ARG(!err, err);
    const bool deform = scene->raw && scene->use_deform && scene->n_dynamic > 0;
    PreFwdParams p;
    p.sc = *scene;
    p.view = *view;
    p.geom = *geom;
    // TMA needs 16-byte aligned global sources; torch allocations are, arbitrary views may not be
    const bool aligned = (((uintptr_t)scene->st.sh_rest | (uintptr_t)scene->dy.sh_rest) & 15u) == 0;
    p.use_tma = aligned ? 1 : 0;
    p.l2_prefetch = rdg_tunable(RDG_TUN_L2_PREFETCH) != 0 ? 1 : 0;
    size_t smem = (RDG_BLOCK * SH_ROW + RDG_NUM_BASIS_MAX * 7) * sizeof(float);
    // B(t) - table rows in shared memory when the whole table fits next to the SH rows with 2 CTAs per SM (T <= 140)
    p.diff_smem = 0;
    if (deform && scene->num_basis == RDG_NUM_BASIS_MAX && rdg_tunable(RDG_TUN_DIFF_SMEM) != 0 &&
        (((uintptr_t)scene->basis_t | (uintptr_t)scene->table) & 15u) == 0) {
        const size_t extra = (size_t)scene->num_times * RDG_DIFF_STRIDE * sizeof(float);
        if (smem + extra <= RDG_PRE_SMEM_MAX) { p.diff_smem = 1; smem += extra; }
    }
    const int64_t chunks = (scene->n_static + RDG_BLOCK - 1) / RDG_BLOCK + (scene->n_dynamic + RDG_BLOCK - 1) / RDG_BLOCK;
    // persistent grid: a multiple of the SM count.  2 CTAs are resident per SM (registers); with the staged difference
    // table every CTA pays for filling it once, so the grid is exactly the resident set
    const int64_t per_sm = p.diff_smem ? 2 : 4;
    const int grid = (int)(chunks < (int64_t)RDG_SM_COUNT * per_sm ? chunks : (int64_t)RDG_SM_COUNT * per_sm);
    cudaStream_t s = (cudaStream_t)stream;
    if (geom->tile_count) {
        const int tiles = ((view->width + RDG_TILE - 1) / RDG_TILE) * ((view->height + RDG_TILE - 1) / RDG_TILE);
        RDG_CUDA(cudaMemsetAsync(geom->tile_count, 0, (size_t)(tiles + 1) * sizeof(uint32_t), s));
    }
    const int rc = scene->raw ? launch_fwd_deg<true>(p, view->sh_degree, grid, smem, s)
                              : launch_fwd_deg<false>(p, view->sh_degree, grid, smem, s);
    if (rc) return rc;
    rdg_count_launches(1);
    return RDG_OK;
}

// ---- several views per launch (rdg_preprocess_fwd_views) ----
//
// Every parameter a Gaussian's footprint and colour depend on except the camera and B(t) is the same in all views: the
// chunk's SH rows are staged, and its geometry, activations, motion coefficients and birth index loaded, ONCE; then each
// view deforms its own copy (c . (B(t_v) - table[t_i])), projects it and colours it with the single-view kernel's device
// functions above.  The table rows are staged in shared memory once for all views when T <= RDG_VIEWS_TABLE_MAX (each
// view's B(t_v) row sits beside them and the difference is formed in registers: the same rounded float as
// rdg_stage_diff's), otherwise each Gaussian gathers its row from global memory as the single-view kernel does.
#define RDG_VIEWS_MAX 8
struct RdgViewCam {
    RdgCam cam;
    float campos[3];
};
// dynamic shared memory without the table: SH rows, B(t) of RDG_VIEWS_MAX views, their cameras
#define RDG_VIEWS_SMEM_BASE \
    ((size_t)(RDG_BLOCK * SH_ROW + RDG_VIEWS_MAX * RDG_NUM_BASIS_MAX * 7) * sizeof(float) + RDG_VIEWS_MAX * sizeof(RdgViewCam))
// largest T whose table rows fit beside them with 2 CTAs per SM: 137
#define RDG_VIEWS_TABLE_MAX ((int)((RDG_PRE_SMEM_MAX - RDG_VIEWS_SMEM_BASE) / (RDG_DIFF_STRIDE * sizeof(float))))

struct PreFwdViewsParams {
    RdgScene sc;
    RdgView view[RDG_VIEWS_MAX];
    RdgGeom geom[RDG_VIEWS_MAX];
    const float* basis_ts;   // [num_views, num_basis, 7]
    int num_views;
    int use_tma;
    int table_smem;          // table rows staged in shared memory
};

template <bool RAW, int DEG>
__global__ void __launch_bounds__(RDG_BLOCK, 2) preprocess_fwd_views_kernel(const PreFwdViewsParams p) {
    extern __shared__ __align__(128) float smem[];
    constexpr int K = (DEG + 1) * (DEG + 1);
    constexpr int NREST = 3 * (K - 1);
    constexpr int BT = RDG_NUM_BASIS_MAX * 7;
    const RdgScene& sc = p.sc;
    const int nv = p.num_views;
    float* sh_s = smem;                                             // [256][SH_ROW]
    float* bt_s = smem + RDG_BLOCK * SH_ROW;                        // [RDG_VIEWS_MAX][BT] B(t_v)
    RdgViewCam* cam_s = reinterpret_cast<RdgViewCam*>(bt_s + RDG_VIEWS_MAX * BT);
    float* table_s = reinterpret_cast<float*>(cam_s + RDG_VIEWS_MAX);  // [T][RDG_DIFF_STRIDE] when p.table_smem
    __shared__ __align__(8) uint64_t bar;

    if ((int)threadIdx.x < nv) {
        const int v = threadIdx.x;
        const RdgView& vw = p.view[v];
        rdg_load_cam(cam_s[v].cam, vw.viewmatrix, vw.projmatrix, vw.tanfovx, vw.tanfovy, vw.width, vw.height);
        rdg_campos(cam_s[v].cam, cam_s[v].campos);
    }
    const bool deform = RAW && sc.use_deform && sc.n_dynamic > 0;
    if (deform) {
        const int row = sc.num_basis * 7;
        for (int e = threadIdx.x; e < nv * row; e += RDG_BLOCK) bt_s[(e / row) * BT + e % row] = p.basis_ts[e];
        if (p.table_smem) {
            const float4* tab4 = reinterpret_cast<const float4*>(sc.table);
            for (int idx = threadIdx.x; idx < sc.num_times * 28; idx += RDG_BLOCK) {
                const int t = idx / 28, q = idx - t * 28;
                *reinterpret_cast<float4*>(table_s + t * RDG_DIFF_STRIDE + 4 * q) = __ldg(tab4 + idx);
            }
        }
    }
    if (threadIdx.x == 0) rdg_mbar_init(&bar, 1);
    __syncthreads();

    const bool use_sh = (sc.colors_precomp == nullptr) && NREST > 0;
    const int64_t cs = (sc.n_static + RDG_BLOCK - 1) / RDG_BLOCK, cd = (sc.n_dynamic + RDG_BLOCK - 1) / RDG_BLOCK;
    uint32_t phase = 0;
    for (int64_t chunk = blockIdx.x; chunk < cs + cd; chunk += gridDim.x) {
        const bool dyn = chunk >= cs;
        const RdgSet& set = dyn ? sc.dy : sc.st;
        const int64_t lbase = (dyn ? chunk - cs : chunk) * RDG_BLOCK;
        const int64_t n_set = dyn ? sc.n_dynamic : sc.n_static;
        const int cnt = (int)min((int64_t)RDG_BLOCK, n_set - lbase);

        // ---- stage this chunk's higher-order SH rows in shared memory (as preprocess_fwd_kernel) ----
        bool tma = false;
        if (use_sh) {
            __syncthreads();  // previous chunk's readers are done with sh_s
            tma = p.use_tma && NREST == SH_ROW && set.sh_rest_stride == SH_ROW && (cnt & 3) == 0;
            if (tma) {
                if (threadIdx.x == 0) {
                    rdg_fence_proxy_async();
                    rdg_bulk_load(sh_s, set.sh_rest + lbase * SH_ROW, (uint32_t)(cnt * SH_ROW * sizeof(float)), &bar);
                }
            } else {
                const int stride = set.sh_rest_stride;
                const float* src = set.sh_rest + lbase * stride;
                for (int e = threadIdx.x; e < cnt * NREST; e += RDG_BLOCK) {
                    const int g = e / NREST, k = e - g * NREST;
                    sh_s[g * SH_ROW + k] = src[(int64_t)g * stride + k];
                }
            }
        }

        const bool valid = (int)threadIdx.x < cnt;
        const int64_t local = lbase + threadIdx.x;
        const int64_t i = (dyn ? sc.n_static : 0) + local;
        RdgAct base;
        float dc0 = 0.f, dc1 = 0.f, dc2 = 0.f;
        if (valid && !sc.colors_precomp) {
            const float* dc = set.sh_dc + local * set.sh_dc_stride;
            dc0 = __ldg(dc); dc1 = __ldg(dc + 1); dc2 = __ldg(dc + 2);
        }
        if (valid) rdg_fetch<RAW, false>(sc, dyn, local, nullptr, base);
        for (int v = 0; v < nv; ++v) {
            const RdgCam& cam = cam_s[v].cam;
            RdgFootprint f;
            RdgAct a = base;
            if (valid) {
                if (deform && dyn) {
                    float d[7];
                    if (p.table_smem) {
                        // the coefficients again from L1 rather than held across the views: no spills at 128 registers
                        const float4* pc4 = reinterpret_cast<const float4*>(sc.motion_coeff + local * RDG_NUM_BASIS_MAX);
                        float c[RDG_NUM_BASIS_MAX];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const float4 w = __ldg(pc4 + q);
                            c[4 * q] = w.x; c[4 * q + 1] = w.y; c[4 * q + 2] = w.z; c[4 * q + 3] = w.w;
                        }
                        rdg_deform_delta_rows(bt_s + v * BT, table_s + a.ti * RDG_DIFF_STRIDE, c, d);
                    } else {
                        rdg_deform_delta(sc, bt_s + v * BT, a.ti, a.c, d);
                    }
                    rdg_apply_deform(sc, d, a);
                }
                rdg_fwd_footprint(p.geom[v], i, cam, a, p.view[0].scale_modifier, f);
            }
            if (v == 0 && use_sh) {
                if (tma) rdg_mbar_wait(&bar, phase & 1u);
                else __syncthreads();
            }
            rdg_fwd_finish<DEG>(p.geom[v], sc, i, valid, f, a, cam_s[v].campos, dc0, dc1, dc2, sh_s + threadIdx.x * SH_ROW);
        }
        if (tma) ++phase;
    }
}

template <bool RAW, int DEG>
static int launch_fwd_views(const PreFwdViewsParams& p, int grid, size_t smem, cudaStream_t s) {
    RDG_CUDA(cudaFuncSetAttribute(preprocess_fwd_views_kernel<RAW, DEG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    preprocess_fwd_views_kernel<RAW, DEG><<<grid, RDG_BLOCK, smem, s>>>(p);
    RDG_CHECK_LAUNCH();
    return RDG_OK;
}

template <bool RAW>
static int launch_fwd_views_deg(const PreFwdViewsParams& p, int deg, int grid, size_t smem, cudaStream_t s) {
    switch (deg) {
        case 0: return launch_fwd_views<RAW, 0>(p, grid, smem, s);
        case 1: return launch_fwd_views<RAW, 1>(p, grid, smem, s);
        case 2: return launch_fwd_views<RAW, 2>(p, grid, smem, s);
        default: return launch_fwd_views<RAW, 3>(p, grid, smem, s);
    }
}

extern "C" int rdg_preprocess_fwd_views(const RdgScene* scene, const float* basis_ts, int32_t num_views, const RdgView* views,
                                        const RdgGeom* geoms, void* stream) {
    RDG_CHECK_ARG(scene && views && geoms, "null argument");
    RDG_CHECK_ARG(num_views >= 1 && num_views <= RDG_VIEWS_MAX, "num_views must be 1..8");
    RDG_CHECK_ARG(scene->basis_t == nullptr, "scene->basis_t must be NULL: each view's B(t) comes from basis_ts");
    const int64_t N = scene->n_static + scene->n_dynamic;
    RDG_CHECK_ARG(N >= 0 && scene->n_static >= 0 && scene->n_dynamic >= 0, "negative count");
    for (int v = 0; v < num_views; ++v) {
        const char* err = view_arg_error(&views[v]);
        RDG_CHECK_ARG(!err, err);
        RDG_CHECK_ARG(views[v].height == views[0].height && views[v].width == views[0].width &&
                          views[v].sh_degree == views[0].sh_degree && views[v].scale_modifier == views[0].scale_modifier,
                      "the views must share height, width, sh_degree and scale_modifier");
    }
    if (N == 0) return RDG_OK;
    for (int v = 0; v < num_views; ++v) RDG_CHECK_ARG(geom_complete(&geoms[v]), "null geometry buffer");
    const char* err = scene_arg_error(scene, views[0].sh_degree, basis_ts);
    RDG_CHECK_ARG(!err, err);
    PreFwdViewsParams p;
    p.sc = *scene;
    for (int v = 0; v < RDG_VIEWS_MAX; ++v) {
        p.view[v] = views[v < num_views ? v : 0];
        p.geom[v] = geoms[v < num_views ? v : 0];
    }
    p.basis_ts = basis_ts;
    p.num_views = num_views;
    p.use_tma = ((((uintptr_t)scene->st.sh_rest | (uintptr_t)scene->dy.sh_rest) & 15u) == 0) ? 1 : 0;
    const bool deform = scene->raw && scene->use_deform && scene->n_dynamic > 0;
    size_t smem = RDG_VIEWS_SMEM_BASE;
    p.table_smem = 0;
    if (deform && scene->num_basis == RDG_NUM_BASIS_MAX && scene->num_times <= RDG_VIEWS_TABLE_MAX &&
        ((uintptr_t)scene->table & 15u) == 0) {
        p.table_smem = 1;
        smem += (size_t)scene->num_times * RDG_DIFF_STRIDE * sizeof(float);
    }
    const int64_t chunks = (scene->n_static + RDG_BLOCK - 1) / RDG_BLOCK + (scene->n_dynamic + RDG_BLOCK - 1) / RDG_BLOCK;
    const int grid = (int)(chunks < (int64_t)RDG_SM_COUNT * 2 ? chunks : (int64_t)RDG_SM_COUNT * 2);   // 2 CTAs per SM
    cudaStream_t s = (cudaStream_t)stream;
    const int tiles = ((views[0].width + RDG_TILE - 1) / RDG_TILE) * ((views[0].height + RDG_TILE - 1) / RDG_TILE);
    for (int v = 0; v < num_views; ++v)
        if (geoms[v].tile_count) RDG_CUDA(cudaMemsetAsync(geoms[v].tile_count, 0, (size_t)(tiles + 1) * sizeof(uint32_t), s));
    const int rc = scene->raw ? launch_fwd_views_deg<true>(p, views[0].sh_degree, grid, smem, s)
                              : launch_fwd_views_deg<false>(p, views[0].sh_degree, grid, smem, s);
    if (rc) return rc;
    rdg_count_launches(1);
    return RDG_OK;
}
