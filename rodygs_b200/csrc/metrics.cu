// Evaluation image metrics: MSE, PSNR, SSIM and MS-SSIM of a batch of image pairs in one pass per scale.
// Definitions are piqa's (what RoDyGSEvaluator.eval and VizScoreEvaluator report), recalled rather than pinned:
// see INTEGRATION.md "Scoring held-out views".  This is NOT the training SSIM of loss.cu: that one zero-pads the
// window over the full image, this one keeps only the valid region (the map is (H-10) x (W-10)) and averages per
// channel; the two give different numbers.
//
// One launch per scale (batch and channel flattened into the grid) + one finalize launch.  A CTA reads a 42x42
// input tile once into shared memory and from it
//   - blurs the five moment planes (x, y, x^2, y^2, xy) separably down to its 32x32 tile of the valid map and sums
//     the SSIM and contrast-structure maps over the tile,
//   - (scale 0) sums (x - y)^2 over the input pixels it owns,
//   - (scales 0..3, MS-SSIM only) writes the 2x2 average pool (ceil mode) of the input pixels it owns: the next
//     scale's input, so that every scale is read from memory once.
// A CTA owns the input rows / columns [32 t, 32 t + 32) of its tile; the last tile of a row or column also owns the
// last 10 inputs behind it, so every input pixel belongs to exactly one CTA.  Tile origins are even, so no 2x2
// pooling window straddles two CTAs.  Per-CTA sums go to fixed workspace slots in float64 and the finalize adds them
// in a fixed order: no float atomics, bit-identical from run to run, and an image's result does not depend on the
// other images of the batch.
#include <math.h>
#include "common.cuh"

#define MT 32                   // valid-map tile edge per CTA
#define MWIN 11                 // Gaussian window
#define MIN_EDGE (MT + MWIN - 1)  // 42: input tile edge
#define MIPITCH 43              // odd row pitch: 32 rows at one column hit 32 banks
#define MHPITCH 33
#define MTHREADS 256
#define MSEG 8                  // outputs per thread, horizontal pass
#define MVSEG 4                 // outputs per thread, vertical pass
#define MSCALES 5
#define MSLOT 3                 // doubles per CTA slot: sum ss, sum cs, sum (x - y)^2

// the normalised 11-tap Gaussian, sigma 1.5, as float32 (the taps of loss_utils.create_window)
__constant__ float c_mtaps[MWIN] = {1.028380124e-03f, 7.598758209e-03f, 3.600077331e-02f, 1.093606874e-01f,
                                    2.130055279e-01f, 2.660117149e-01f, 2.130055279e-01f, 1.093606874e-01f,
                                    3.600077331e-02f, 7.598758209e-03f, 1.028380124e-03f};

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One scale of one plane tile.  x, y: [planes, H, W]; px, py: [planes, ceil(H/2), ceil(W/2)] or NULL (last scale);
// part[blockIdx.x] <- (sum ss, sum cs, sum (x - y)^2 if want_sq).
__global__ void __launch_bounds__(MTHREADS) metrics_scale_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                                 int H, int W, int tiles_x, int tiles_y,
                                                                 float* __restrict__ px, float* __restrict__ py, int want_sq,
                                                                 float C1, float C2, double* __restrict__ part) {
    __shared__ float in[2][MIN_EDGE][MIPITCH];
    __shared__ float hz[5][MIN_EDGE][MHPITCH];
    __shared__ double red[MSLOT][MTHREADS / 32];
    const int tiles = tiles_x * tiles_y;
    const int p = blockIdx.x / tiles, tile = blockIdx.x - p * tiles;
    const int tx = tile % tiles_x, ty = tile / tiles_x;
    const int x0 = tx * MT, y0 = ty * MT;
    const size_t plane = (size_t)p * H * W;
    for (int idx = threadIdx.x; idx < MIN_EDGE * MIN_EDGE; idx += MTHREADS) {
        const int r = idx / MIN_EDGE, c = idx - r * MIN_EDGE;
        const int yy = y0 + r, xx = x0 + c;
        float a = 0.f, b = 0.f;
        if (xx < W && yy < H) { a = x[plane + (size_t)yy * W + xx]; b = y[plane + (size_t)yy * W + xx]; }
        in[0][r][c] = a;
        in[1][r][c] = b;
    }
    __syncthreads();
    // Moments are taken about a value of the tile (always in bounds: y0 <= H - 11, x0 <= W - 11).  Variance and
    // covariance do not change under the shift, and in flat regions E[x^2] - E[x]^2 no longer cancels in float32.
    const float cx = in[0][MWIN / 2][MWIN / 2], cy = in[1][MWIN / 2][MWIN / 2];
    if (threadIdx.x < MIN_EDGE * (MT / MSEG)) {
        const int r = threadIdx.x % MIN_EDGE, s = threadIdx.x / MIN_EDGE;
        float a[5][MSEG];
#pragma unroll
        for (int q = 0; q < 5; ++q)
#pragma unroll
            for (int i = 0; i < MSEG; ++i) a[q][i] = 0.f;
#pragma unroll
        for (int k = 0; k < MSEG + MWIN - 1; ++k) {
            const float xv = in[0][r][s * MSEG + k] - cx, yv = in[1][r][s * MSEG + k] - cy;
            const float xx = xv * xv, yy = yv * yv, xy = xv * yv;
#pragma unroll
            for (int i = 0; i < MSEG; ++i) {
                const int tap = k - i;
                if (tap >= 0 && tap < MWIN) {
                    const float w = c_mtaps[tap];
                    a[0][i] = __fmaf_rn(w, xv, a[0][i]);
                    a[1][i] = __fmaf_rn(w, yv, a[1][i]);
                    a[2][i] = __fmaf_rn(w, xx, a[2][i]);
                    a[3][i] = __fmaf_rn(w, yy, a[3][i]);
                    a[4][i] = __fmaf_rn(w, xy, a[4][i]);
                }
            }
        }
#pragma unroll
        for (int q = 0; q < 5; ++q)
#pragma unroll
            for (int i = 0; i < MSEG; ++i) hz[q][r][s * MSEG + i] = a[q][i];
    }
    __syncthreads();
    const int c = threadIdx.x % MT, vs = threadIdx.x / MT;
    float o[5][MVSEG];
#pragma unroll
    for (int q = 0; q < 5; ++q)
#pragma unroll
        for (int i = 0; i < MVSEG; ++i) o[q][i] = 0.f;
#pragma unroll
    for (int k = 0; k < MVSEG + MWIN - 1; ++k) {
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            const float v = hz[q][vs * MVSEG + k][c];
#pragma unroll
            for (int i = 0; i < MVSEG; ++i) {
                const int tap = k - i;
                if (tap >= 0 && tap < MWIN) o[q][i] = __fmaf_rn(c_mtaps[tap], v, o[q][i]);
            }
        }
    }
    double acc[MSLOT] = {0.0, 0.0, 0.0};
    const int Hv = H - (MWIN - 1), Wv = W - (MWIN - 1);
    if (x0 + c < Wv) {
#pragma unroll
        for (int i = 0; i < MVSEG; ++i) {
            if (y0 + vs * MVSEG + i < Hv) {
                const float mx = cx + o[0][i], my = cy + o[1][i];
                const float sxx = o[2][i] - o[0][i] * o[0][i], syy = o[3][i] - o[1][i] * o[1][i];
                const float sxy = o[4][i] - o[0][i] * o[1][i];
                const float cs = (2.f * sxy + C2) / (sxx + syy + C2);
                const float ss = (2.f * mx * my + C1) / (mx * mx + my * my + C1) * cs;
                acc[0] += (double)ss;
                acc[1] += (double)cs;
            }
        }
    }
    // the input pixels this CTA owns
    const int ox1 = tx == tiles_x - 1 ? W : x0 + MT, oy1 = ty == tiles_y - 1 ? H : y0 + MT;
    const int ow = ox1 - x0, oh = oy1 - y0;
    if (want_sq) {
        for (int idx = threadIdx.x; idx < ow * oh; idx += MTHREADS) {
            const int r = idx / ow, cc = idx - r * ow;
            const double d = (double)(in[0][r][cc] - in[1][r][cc]);
            acc[2] += d * d;
        }
    }
    if (px) {
        // avg_pool2d(kernel 2, stride 2, ceil_mode=True, padding 0): a window that hangs over the last row / column
        // averages its in-bounds pixels only; float sum in row-major window order, then one division (as PyTorch does)
        const int Hp = (H + 1) / 2, Wp = (W + 1) / 2;
        const int pw = (ow + 1) / 2, ph = (oh + 1) / 2;
        const size_t pplane = (size_t)p * Hp * Wp;
        for (int idx = threadIdx.x; idx < pw * ph; idx += MTHREADS) {
            const int pr = idx / pw, pc = idx - pr * pw;
            const int r = 2 * pr, cc = 2 * pc;
            const bool r1 = y0 + r + 1 < H, c1 = x0 + cc + 1 < W;
            float sx = in[0][r][cc], sy = in[1][r][cc];
            if (c1) { sx += in[0][r][cc + 1]; sy += in[1][r][cc + 1]; }
            if (r1) { sx += in[0][r + 1][cc]; sy += in[1][r + 1][cc]; }
            if (r1 && c1) { sx += in[0][r + 1][cc + 1]; sy += in[1][r + 1][cc + 1]; }
            const float cnt = (float)((1 + (int)c1) * (1 + (int)r1));
            const size_t o_idx = pplane + (size_t)(y0 / 2 + pr) * Wp + (x0 / 2 + pc);
            px[o_idx] = sx / cnt;
            py[o_idx] = sy / cnt;
        }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 0; k < MSLOT; ++k) {
        const double v = warp_sum_d(acc[k]);
        if (lane == 0) red[k][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < MSLOT) {
        double t = 0.0;
        for (int w = 0; w < MTHREADS / 32; ++w) t += red[threadIdx.x][w];
        part[(size_t)blockIdx.x * MSLOT + threadIdx.x] = t;
    }
}

struct MetricsFinal {
    const double* part[MSCALES];   // per scale: [planes][tiles] slots
    int tiles[MSCALES];
    double valid[MSCALES];         // (H_s - 10) (W_s - 10)
    int nscales, channels;
    double n_all;                  // C H W
    double range2;
};

// Sum of field k over `count` consecutive slots, in a fixed order (strided per thread, then a fixed tree).
__device__ double block_sum_slots(const double* __restrict__ base, int count, int k, double* sh) {
    double t = 0.0;
    for (int i = threadIdx.x; i < count; i += MTHREADS) t += base[(size_t)i * MSLOT + k];
    sh[threadIdx.x] = t;
    __syncthreads();
    for (int s = MTHREADS / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
        __syncthreads();
    }
    const double r = sh[0];
    __syncthreads();
    return r;
}

// One CTA per image: out[b] = (mse, psnr, ssim, ms_ssim), float64 arithmetic.
__global__ void __launch_bounds__(MTHREADS) metrics_finalize_kernel(MetricsFinal f, float* __restrict__ out) {
    __shared__ double sh[MTHREADS];
    const double wts[MSCALES] = {0.0448, 0.2856, 0.3001, 0.2363, 0.1333};
    const int b = blockIdx.x;
    double sq = 0.0, ssim = 0.0, ms = 0.0;
    for (int c = 0; c < f.channels; ++c) {
        const size_t p = (size_t)b * f.channels + c;
        const double* base0 = f.part[0] + p * f.tiles[0] * MSLOT;
        sq += block_sum_slots(base0, f.tiles[0], 2, sh);
        ssim += block_sum_slots(base0, f.tiles[0], 0, sh) / f.valid[0];
        if (f.nscales == MSCALES) {
            double m = 1.0;
            for (int s = 0; s < MSCALES; ++s) {
                const double* base = f.part[s] + p * f.tiles[s] * MSLOT;
                const int k = s == MSCALES - 1 ? 0 : 1;          // cs at scales 0..3, ss at the last
                const double v = block_sum_slots(base, f.tiles[s], k, sh) / f.valid[s];
                m *= pow(v < 0.0 ? 0.0 : v, wts[s]);             // relu (NaN propagates)
            }
            ms += m;
        }
    }
    if (threadIdx.x == 0) {
        const double mse = sq / f.n_all;
        out[b * 4 + 0] = (float)mse;
        out[b * 4 + 1] = (float)(10.0 * log10(f.range2 / (mse + 1e-8)));
        out[b * 4 + 2] = (float)(ssim / f.channels);
        out[b * 4 + 3] = f.nscales == MSCALES ? (float)(ms / f.channels) : __int_as_float(0x7fc00000);
    }
}

struct MetricsLayout {
    int nscales;
    int H[MSCALES], W[MSCALES], tx[MSCALES], ty[MSCALES];
    int64_t part_off[MSCALES], pool_off[MSCALES];   // pool_off[s]: x plane of scale s >= 1 (y follows)
    int64_t total;
};

static int metrics_check_dims(const char* fn, int32_t batch, int32_t channels, int32_t height, int32_t width) {
    if (batch < 1) { rdg_set_error("%s: batch must be >= 1 (got %d)", fn, batch); return RDG_E_ARG; }
    if (channels < 1) { rdg_set_error("%s: channels must be >= 1 (got %d)", fn, channels); return RDG_E_ARG; }
    if (height < MWIN) { rdg_set_error("%s: height must be >= 11, the SSIM window (got %d)", fn, height); return RDG_E_ARG; }
    if (width < MWIN) { rdg_set_error("%s: width must be >= 11, the SSIM window (got %d)", fn, width); return RDG_E_ARG; }
    return RDG_OK;
}

static int metrics_layout(const char* fn, int32_t batch, int32_t channels, int32_t height, int32_t width, MetricsLayout* L) {
    const int rc = metrics_check_dims(fn, batch, channels, height, width);
    if (rc != RDG_OK) return rc;
    // MS-SSIM needs every one of the 5 scales to hold the window: ceil(H / 16), ceil(W / 16) >= 11
    const bool ms = (height + 15) / 16 >= MWIN && (width + 15) / 16 >= MWIN;
    L->nscales = ms ? MSCALES : 1;
    const int64_t planes = (int64_t)batch * channels;
    int64_t off = 0;
    int h = height, w = width;
    for (int s = 0; s < L->nscales; ++s) {
        L->H[s] = h;
        L->W[s] = w;
        L->tx[s] = rdg_div_up(w - (MWIN - 1), MT);
        L->ty[s] = rdg_div_up(h - (MWIN - 1), MT);
        const int64_t ctas = planes * L->tx[s] * L->ty[s];
        if (ctas > INT32_MAX) { rdg_set_error("%s: batch * channels * tiles exceeds the grid", fn); return RDG_E_ARG; }
        L->part_off[s] = off;
        off += rdg_align_up(ctas * MSLOT * (int64_t)sizeof(double), 256);
        h = (h + 1) / 2;
        w = (w + 1) / 2;
    }
    L->pool_off[0] = -1;
    for (int s = 1; s < L->nscales; ++s) {
        L->pool_off[s] = off;
        off += 2 * rdg_align_up(planes * L->H[s] * L->W[s] * (int64_t)sizeof(float), 256);
    }
    L->total = off;
    return RDG_OK;
}

extern "C" int64_t rdg_image_metrics_workspace_bytes(int32_t batch, int32_t channels, int32_t height, int32_t width) {
    MetricsLayout L;
    const int rc = metrics_layout(__func__, batch, channels, height, width, &L);
    return rc != RDG_OK ? rc : L.total;
}

extern "C" int rdg_image_metrics(const float* pred, const float* gt, int32_t batch, int32_t channels, int32_t height,
                                 int32_t width, float value_range, float* out, void* workspace, int64_t workspace_bytes,
                                 void* stream) {
    RDG_CHECK_ARG(pred, "pred is NULL");
    RDG_CHECK_ARG(gt, "gt is NULL");
    RDG_CHECK_ARG(out, "out is NULL");
    RDG_CHECK_ARG(workspace, "workspace is NULL");
    MetricsLayout L;
    const int rc = metrics_layout(__func__, batch, channels, height, width, &L);
    if (rc != RDG_OK) return rc;
    RDG_CHECK_ARG(value_range > 0.0f && isfinite(value_range), "value_range must be a finite value > 0");
    RDG_CHECK_ARG(workspace_bytes >= L.total, "workspace_bytes is smaller than rdg_image_metrics_workspace_bytes()");
    RDG_CHECK_ARG(((uintptr_t)workspace & 15) == 0, "workspace must be 16-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    const int64_t planes = (int64_t)batch * channels;
    const double r = (double)value_range;
    const float C1 = (float)((0.01 * r) * (0.01 * r)), C2 = (float)((0.03 * r) * (0.03 * r));
    MetricsFinal f = {};
    const float* xs = pred;
    const float* ys = gt;
    for (int sc = 0; sc < L.nscales; ++sc) {
        float* px = nullptr;
        float* py = nullptr;
        if (sc + 1 < L.nscales) {
            px = (float*)(ws + L.pool_off[sc + 1]);
            py = (float*)(ws + L.pool_off[sc + 1] + rdg_align_up(planes * L.H[sc + 1] * L.W[sc + 1] * (int64_t)sizeof(float), 256));
        }
        double* part = (double*)(ws + L.part_off[sc]);
        const int tiles = L.tx[sc] * L.ty[sc];
        metrics_scale_kernel<<<(unsigned)(planes * tiles), MTHREADS, 0, s>>>(xs, ys, L.H[sc], L.W[sc], L.tx[sc], L.ty[sc], px, py,
                                                                              sc == 0 ? 1 : 0, C1, C2, part);
        RDG_CHECK_LAUNCH();
        f.part[sc] = part;
        f.tiles[sc] = tiles;
        f.valid[sc] = (double)(L.H[sc] - (MWIN - 1)) * (double)(L.W[sc] - (MWIN - 1));
        xs = px;
        ys = py;
    }
    f.nscales = L.nscales;
    f.channels = channels;
    f.n_all = (double)channels * height * width;
    f.range2 = r * r;
    metrics_finalize_kernel<<<batch, MTHREADS, 0, s>>>(f, out);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(L.nscales + 1);
    return RDG_OK;
}

// ---- masked metrics: DyCheck's mPSNR / mSSIM over a covisibility mask ----------------------------------------------------
// Definitions (recalled, unpinned: INTEGRATION.md "Scoring held-out views") for mask m [H, W] shared by the channels:
//   mmse = sum m (x - y)^2 / (C sum m), mpsnr = 10 log10(R^2 / mmse) (no epsilon: an empty mask gives NaN, mmse = 0 +inf);
//   mssim = mean over all C (H-10) (W-10) positions of the SSIM map of a two-stage "valid" partial convolution
//     stage 1 (width):  n1 = sum_k m_k,  P1(z) = n1 != 0 ? 11 sum_k g_k m_k z_k / n1 : 0,  v1 = (n1 != 0)
//     stage 2 (height): n2 = sum_k v1_k, P(z)  = n2 != 0 ? 11 sum_k g_k v1_k P1(z)_k / n2 : 0
//   with sigma_xx = max(0, P(x^2) - P(x)^2), sigma_xy = sign(s) min(sqrt(sigma_xx sigma_yy), |s|), s = P(xy) - P(x) P(y).
//   A window without a covisible pixel has mu = sigma = 0 and a map value of exactly 1.
// One launch over (image, channel, tile) with the tiling and pixel ownership of metrics_scale_kernel, then a one-CTA-per-image
// finalize; float64 partials in fixed slots summed in a fixed order, so the result is bit-identical from run to run and an
// image's row does not depend on the rest of the batch.
//
// Precision.  P does not preserve constants (P(1) != 1 next to masked-out pixels), so the tile's moments are taken about a
// covisible value c of the tile and sigma_xx = [P(x'^2) - P(x')^2] + 2c P(x') D + c^2 (1 - D) D with x' = x - c and
// D = 1 - P(1).  D is carried as its own plane, built from the masked-OUT weights only:
//   1 - P1(1) = 11 sum_k (g_k - 1/11) (1 - m_k) / n1,   1 - P(1) = 11 [sum_k g_k (1 - P1(1))_k v1_k + sum_k (g_k - 1/11)(1 - v1_k)] / n2
// (sum_k (g_k - 1/11) = 0), so D is exactly 0 wherever the window is fully covisible and a flat region keeps sigma = 0
// instead of float32 noise of order c^2 * 1e-7.  Masked-out and out-of-image pixels are replaced by 0 on load (a select,
// so NaN / Inf under the mask never propagate) and c is taken from a covisible pixel: masked-out values change no bit.

#define MPLANES 7               // P1 of x', y', x'^2, y'^2, x'y', then 1 - P1(1) and v1

// g_k - 1/11 of the float64-normalised taps, rounded to float32
__constant__ float c_mdef[MWIN] = {-8.988071233e-02f, -8.331033587e-02f, -5.490832031e-02f, 1.845159940e-02f,
                                   1.220964491e-01f,  1.751026362e-01f,  1.220964491e-01f,  1.845159940e-02f,
                                   -5.490832031e-02f, -8.331033587e-02f, -8.988071233e-02f};

struct MaskedSmem {
    float in[3][MIN_EDGE][MIPITCH];        // x, y, m (0, 0, 0 where masked out or outside the image)
    float hz[MPLANES][MIN_EDGE][MHPITCH];  // stage 1 output
    double red[MSLOT][MTHREADS / 32];
    int ref;                               // key of the tile's reference pixel (INT_MAX: no covisible pixel)
};

// x, y: [planes, H, W]; m: [planes / C, H, W]; part[blockIdx.x] <- (sum map, sum m (x - y)^2, sum m) over the tile.
__global__ void __launch_bounds__(MTHREADS) masked_metrics_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                                  const float* __restrict__ m, int C, int H, int W,
                                                                  int tiles_x, int tiles_y, float C1, float C2,
                                                                  double* __restrict__ part) {
    extern __shared__ __align__(16) unsigned char masked_smem[];
    MaskedSmem& sm = *reinterpret_cast<MaskedSmem*>(masked_smem);
    const int tiles = tiles_x * tiles_y;
    const int p = blockIdx.x / tiles, tile = blockIdx.x - p * tiles;
    const int tx = tile % tiles_x, ty = tile / tiles_x;
    const int x0 = tx * MT, y0 = ty * MT;
    const size_t plane = (size_t)p * H * W, mplane = (size_t)(p / C) * H * W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) sm.ref = INT_MAX;
    // reference pixel: the covisible pixel nearest the tile's centre, ties to the lower row-major index
    int key = INT_MAX;
    for (int idx = threadIdx.x; idx < MIN_EDGE * MIN_EDGE; idx += MTHREADS) {
        const int r = idx / MIN_EDGE, c = idx - r * MIN_EDGE;
        const int yy = y0 + r, xx = x0 + c;
        float a = 0.f, b = 0.f, w = 0.f;
        if (xx < W && yy < H) {
            const float mv = m[mplane + (size_t)yy * W + xx];
            if (mv != 0.f) {
                w = mv;
                a = x[plane + (size_t)yy * W + xx];
                b = y[plane + (size_t)yy * W + xx];
                key = min(key, (abs(2 * r - (MIN_EDGE - 1)) + abs(2 * c - (MIN_EDGE - 1))) * 2048 + idx);
            }
        }
        sm.in[0][r][c] = a;
        sm.in[1][r][c] = b;
        sm.in[2][r][c] = w;
    }
    key = __reduce_min_sync(0xffffffffu, key);
    __syncthreads();
    if (lane == 0) atomicMin(&sm.ref, key);
    __syncthreads();
    float cx = 0.f, cy = 0.f;
    if (sm.ref != INT_MAX) {
        const int i = sm.ref & 2047, r = i / MIN_EDGE;
        cx = sm.in[0][r][i - r * MIN_EDGE];
        cy = sm.in[1][r][i - r * MIN_EDGE];
    }
    // stage 1, along the width: 42 rows x 32 outputs
    if (threadIdx.x < MIN_EDGE * (MT / MSEG)) {
        const int r = threadIdx.x % MIN_EDGE, s = threadIdx.x / MIN_EDGE;
        float a[5][MSEG], n[MSEG], e[MSEG];
#pragma unroll
        for (int i = 0; i < MSEG; ++i) {
#pragma unroll
            for (int q = 0; q < 5; ++q) a[q][i] = 0.f;
            n[i] = 0.f;
            e[i] = 0.f;
        }
#pragma unroll
        for (int k = 0; k < MSEG + MWIN - 1; ++k) {
            const int cc = s * MSEG + k;
            const float w = sm.in[2][r][cc];
            const float xv = sm.in[0][r][cc] - cx, yv = sm.in[1][r][cc] - cy;
            const float wx = w * xv, wy = w * yv;
            const float v[5] = {wx, wy, wx * xv, wy * yv, wx * yv};
            const float u = 1.f - w;
#pragma unroll
            for (int i = 0; i < MSEG; ++i) {
                const int tap = k - i;
                if (tap >= 0 && tap < MWIN) {
                    const float g = c_mtaps[tap];
#pragma unroll
                    for (int q = 0; q < 5; ++q) a[q][i] = __fmaf_rn(g, v[q], a[q][i]);
                    n[i] += w;
                    e[i] = __fmaf_rn(c_mdef[tap], u, e[i]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < MSEG; ++i) {
            const bool ok = n[i] != 0.f;
            const float inv = 11.f / n[i];
#pragma unroll
            for (int q = 0; q < 5; ++q) sm.hz[q][r][s * MSEG + i] = ok ? a[q][i] * inv : 0.f;
            sm.hz[5][r][s * MSEG + i] = ok ? e[i] * inv : 0.f;
            sm.hz[6][r][s * MSEG + i] = ok ? 1.f : 0.f;
        }
    }
    __syncthreads();
    // stage 2, along the height: 32 columns x 32 outputs
    const int c = threadIdx.x % MT, vs = threadIdx.x / MT;
    float o[6][MVSEG], n2[MVSEG];
#pragma unroll
    for (int i = 0; i < MVSEG; ++i) {
#pragma unroll
        for (int q = 0; q < 6; ++q) o[q][i] = 0.f;
        n2[i] = 0.f;
    }
#pragma unroll
    for (int k = 0; k < MVSEG + MWIN - 1; ++k) {
        const int row = vs * MVSEG + k;
        float v[6];
#pragma unroll
        for (int q = 0; q < 6; ++q) v[q] = sm.hz[q][row][c];
        const float valid = sm.hz[6][row][c], u = 1.f - valid;
#pragma unroll
        for (int i = 0; i < MVSEG; ++i) {
            const int tap = k - i;
            if (tap >= 0 && tap < MWIN) {
                const float g = c_mtaps[tap];
#pragma unroll
                for (int q = 0; q < 6; ++q) o[q][i] = __fmaf_rn(g, v[q], o[q][i]);
                o[5][i] = __fmaf_rn(c_mdef[tap], u, o[5][i]);
                n2[i] += valid;
            }
        }
    }
    double acc[MSLOT] = {0.0, 0.0, 0.0};
    const int Hv = H - (MWIN - 1), Wv = W - (MWIN - 1);
    if (x0 + c < Wv) {
#pragma unroll
        for (int i = 0; i < MVSEG; ++i) {
            if (y0 + vs * MVSEG + i < Hv) {
                const bool ok = n2[i] != 0.f;
                const float inv = 11.f / n2[i];
                const float ux = ok ? o[0][i] * inv : 0.f, uy = ok ? o[1][i] * inv : 0.f;
                const float pxx = ok ? o[2][i] * inv : 0.f, pyy = ok ? o[3][i] * inv : 0.f, pxy = ok ? o[4][i] * inv : 0.f;
                const float D = ok ? o[5][i] * inv : 1.f, P1 = 1.f - D;
                const float mx = ux + cx * P1, my = uy + cy * P1;
                const float sxx = fmaxf((pxx - ux * ux) + D * cx * (2.f * ux + cx * P1), 0.f);
                const float syy = fmaxf((pyy - uy * uy) + D * cy * (2.f * uy + cy * P1), 0.f);
                const float s = (pxy - ux * uy) + D * (cy * ux + cx * uy + cx * cy * P1);
                const float sxy = copysignf(fminf(sqrtf(sxx * syy), fabsf(s)), s);
                const float map = ((2.f * mx * my + C1) * (2.f * sxy + C2)) / ((mx * mx + my * my + C1) * (sxx + syy + C2));
                acc[0] += (double)map;
            }
        }
    }
    // the input pixels this CTA owns
    const int ox1 = tx == tiles_x - 1 ? W : x0 + MT, oy1 = ty == tiles_y - 1 ? H : y0 + MT;
    const int ow = ox1 - x0, oh = oy1 - y0;
    for (int idx = threadIdx.x; idx < ow * oh; idx += MTHREADS) {
        const int r = idx / ow, cc = idx - r * ow;
        const double d = (double)sm.in[0][r][cc] - (double)sm.in[1][r][cc], w = (double)sm.in[2][r][cc];
        acc[1] += w * (d * d);
        acc[2] += w;
    }
#pragma unroll
    for (int k = 0; k < MSLOT; ++k) {
        const double v = warp_sum_d(acc[k]);
        if (lane == 0) sm.red[k][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < MSLOT) {
        double t = 0.0;
        for (int w = 0; w < MTHREADS / 32; ++w) t += sm.red[threadIdx.x][w];
        part[(size_t)blockIdx.x * MSLOT + threadIdx.x] = t;
    }
}

// One CTA per image: out[b] = (mmse, mpsnr, mssim), float64 arithmetic.  The mask sum is channel 0's (every channel's
// CTAs sum the same mask).
__global__ void __launch_bounds__(MTHREADS) masked_metrics_finalize_kernel(const double* __restrict__ part, int tiles,
                                                                           int channels, double valid, double range2,
                                                                           float* __restrict__ out) {
    __shared__ double sh[MTHREADS];
    const int b = blockIdx.x;
    const double* img = part + (size_t)b * channels * tiles * MSLOT;
    double sq = 0.0, ssim = 0.0;
    for (int c = 0; c < channels; ++c) {
        const double* base = img + (size_t)c * tiles * MSLOT;
        sq += block_sum_slots(base, tiles, 1, sh);
        ssim += block_sum_slots(base, tiles, 0, sh) / valid;
    }
    const double msum = block_sum_slots(img, tiles, 2, sh);
    if (threadIdx.x == 0) {
        const double mse = sq / (channels * msum);
        out[b * 3 + 0] = (float)mse;
        out[b * 3 + 1] = (float)(10.0 * log10(range2 / mse));
        out[b * 3 + 2] = (float)(ssim / channels);
    }
}

static int masked_layout(const char* fn, int32_t batch, int32_t channels, int32_t height, int32_t width, int* tiles_x,
                         int* tiles_y, int64_t* total) {
    const int rc = metrics_check_dims(fn, batch, channels, height, width);
    if (rc != RDG_OK) return rc;
    *tiles_x = rdg_div_up(width - (MWIN - 1), MT);
    *tiles_y = rdg_div_up(height - (MWIN - 1), MT);
    const int64_t ctas = (int64_t)batch * channels * *tiles_x * *tiles_y;
    if (ctas > INT32_MAX) { rdg_set_error("%s: batch * channels * tiles exceeds the grid", fn); return RDG_E_ARG; }
    *total = rdg_align_up(ctas * MSLOT * (int64_t)sizeof(double), 256);
    return RDG_OK;
}

extern "C" int64_t rdg_masked_image_metrics_workspace_bytes(int32_t batch, int32_t channels, int32_t height, int32_t width) {
    int tx, ty;
    int64_t total;
    const int rc = masked_layout(__func__, batch, channels, height, width, &tx, &ty, &total);
    return rc != RDG_OK ? rc : total;
}

extern "C" int rdg_masked_image_metrics(const float* pred, const float* gt, const float* mask, int32_t batch, int32_t channels,
                                        int32_t height, int32_t width, float value_range, float* out, void* workspace,
                                        int64_t workspace_bytes, void* stream) {
    RDG_CHECK_ARG(pred, "pred is NULL");
    RDG_CHECK_ARG(gt, "gt is NULL");
    RDG_CHECK_ARG(mask, "mask is NULL");
    RDG_CHECK_ARG(out, "out is NULL");
    RDG_CHECK_ARG(workspace, "workspace is NULL");
    int tx, ty;
    int64_t total;
    const int rc = masked_layout(__func__, batch, channels, height, width, &tx, &ty, &total);
    if (rc != RDG_OK) return rc;
    RDG_CHECK_ARG(value_range > 0.0f && isfinite(value_range), "value_range must be a finite value > 0");
    RDG_CHECK_ARG(workspace_bytes >= total, "workspace_bytes is smaller than rdg_masked_image_metrics_workspace_bytes()");
    RDG_CHECK_ARG(((uintptr_t)workspace & 15) == 0, "workspace must be 16-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    const double r = (double)value_range;
    const float C1 = (float)((0.01 * r) * (0.01 * r)), C2 = (float)((0.03 * r) * (0.03 * r));
    double* part = (double*)workspace;
    const size_t smem = sizeof(MaskedSmem);
    RDG_CUDA(cudaFuncSetAttribute(masked_metrics_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    masked_metrics_kernel<<<(unsigned)((int64_t)batch * channels * tx * ty), MTHREADS, smem, s>>>(pred, gt, mask, channels, height,
                                                                                                  width, tx, ty, C1, C2, part);
    RDG_CHECK_LAUNCH();
    masked_metrics_finalize_kernel<<<batch, MTHREADS, 0, s>>>(part, tx * ty, channels,
                                                              (double)(height - (MWIN - 1)) * (double)(width - (MWIN - 1)),
                                                              r * r, out);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(2);
    return RDG_OK;
}
