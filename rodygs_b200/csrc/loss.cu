// Fused photometric loss  w_l1 * L1 + w_dssim * (1 - SSIM)  with its gradient, the
// Pearson depth regulariser over boxes, and a flat fused Adam step.
// SURVEY.md §8 rows a11, a12 (+ f1); spec == oracle/loss_oracle.py, which is pinned
// against /root/reference/src/utils/loss_utils.py by tests/golden/losses.npz.
//
// SSIM: 11-tap separable Gaussian (sigma 1.5, zero padding 5, per channel).  Pass 1
// blurs (x, y, x^2, y^2, xy) of a 32x32 tile from a 42x42 halo in shared memory, forms
// the SSIM map and its three partial-derivative maps; pass 2 blurs those maps and
// applies the chain rule.  24 B/px read + 36 B/px maps written, then 36 + 24 B/px read +
// 12 B/px written (the reference's conv2d chain moves ~700 B/px).  The global Pearson
// depth statistics and the alpha regulariser ride on the channel-0 CTAs of pass 1, their
// gradients on pass 2, so the whole loss stage is three launches.  The LOCAL Pearson term (LocalPearsonDepthLoss,
// /root/reference/src/trainer/losses.py:132-182: ~60 random 128x128 boxes at 1080p, a Python loop of ~25 kernels each in
// the reference) rides along as well: a channel-0 CTA of pass 1 adds its pixels to the statistics of the boxes that
// overlap its tile (0.7 boxes per tile on average), the finalize kernel turns them into per-box coefficients, and pass
// 2 adds every covering box's term to the pixel's dL/ddepth - no atomics on the gradient, no extra pass over the image.
#include <math.h>
#include "common.cuh"

#define ST 32                  // output tile: ST x ST pixels per CTA and channel
#define HALO 5
#define SHL (ST + 2 * HALO)    // 42: halo tile edge
#define IPITCH 43              // halo-tile row pitch; odd, so 32 consecutive rows at one column hit 32 banks
#define HPITCH 33              // row pitch of the horizontally blurred planes
#define LTHREADS 256
#define SEG 8                  // outputs per thread, horizontal pass (sliding window of SEG + 10 inputs in registers)
#define VSEG 4                 // outputs per thread, vertical pass

// /root/reference/src/utils/loss_utils.py:34-41: float32 taps exp(-(i-5)^2 / (2*1.5^2)) / sum,
// evaluated the way the reference does (torch.Tensor of Python floats, divided by its float32 sum).
__constant__ float c_taps[11] = {1.028380124e-03f, 7.598758209e-03f, 3.600077331e-02f, 1.093606874e-01f,
                                 2.130055279e-01f, 2.660117149e-01f, 2.130055279e-01f, 1.093606874e-01f,
                                 3.600077331e-02f, 7.598758209e-03f, 1.028380124e-03f};

// Header of the loss workspace (256 bytes reserved): running sums and the Pearson gradient coefficients.
struct LossHdr {
    double sums[8];   // 0 ssim, 1 |x-y|, 2..6 depth: sum p, g, pp, gg, pg, 7 sum(1 - alpha)
    float coef[8];    // 0 mean g, 1 mean p, 2 d/d(g - mg), 3 d/d(p - mp), 5 rounding correction of the two float means
                      // (dL/ddepth = c2 (g-mg) + c3 (p-mp) + c5), 4 dL/dalpha
    double local_sum; // sum over the boxes of (1 - Pearson_b)
};
#define LOCAL_BOXES_MAX 256
// local-box scratch behind the derivative maps: 8 doubles of statistics + 4 floats of coefficients per box
struct __align__(16) LocalBox {
    float coef[4];    // mean g, mean p, d/d(g - mg), d/d(p - mp), weight included (read as one float4)
    double st[5];     // sum p, g, pp, gg, pg over the box
    float c0;         // rounding correction of the two float means (see pearson_coef_correction)
    int pad;
};
static_assert(sizeof(LocalBox) == 64, "LocalBox layout");

// The gradient of a Pearson term is applied per pixel as c_g (g - mean g) + c_p (p - mean p) with both means rounded to
// float.  Their rounding error is a constant offset over the box that the exact gradient does not have (it sums to zero
// over the box), and c_p grows as 1 / std(p): in a nearly flat box it swamped the per-pixel values.  This constant,
// formed in double, cancels the offset.
__device__ __forceinline__ float pearson_coef_correction(double cg, double mg, double cp, double mp) {
    return (float)(-(cg * (mg - (double)(float)mg) + cp * (mp - (double)(float)mp)));
}

// The local Pearson boxes that overlap the 32x32 tile at (tx0, ty0), in box order, into near[] (call from warp 0; ballot
// compaction, so that per-pixel sums over the list keep one order).  A 128x128 box overlaps ~1 % of the tiles: every thread
// testing all ~60 boxes itself cost 12 M warp instructions per pass (ncu r02).
__device__ __forceinline__ int boxes_near_tile(const int4* __restrict__ boxes, int n_boxes, int tx0, int ty0, int* near) {
    int cnt = 0;
    for (int base = 0; base < n_boxes; base += 32) {
        const int b = base + (int)threadIdx.x;
        bool hit = false;
        if (b < n_boxes) {
            const int4 bx = boxes[b];
            hit = !(bx.x >= ty0 + ST || bx.x + bx.z <= ty0 || bx.y >= tx0 + ST || bx.y + bx.w <= tx0);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (hit) near[cnt + __popc(bal & ((1u << threadIdx.x) - 1u))] = b;
        cnt += __popc(bal);
    }
    return cnt;
}

// Separable 11-tap blur of an SHL x SHL halo tile down to ST x ST, register-tiled: the horizontal pass
// gives every thread one row and SEG adjacent outputs (each input is loaded once and used for up to 11
// taps x NQ planes from registers), the vertical pass one column and VSEG outputs.  12 FMA per shared-memory
// load instead of 1 - the first version of this kernel was LSU bound (ncu r01).
template <int NQ>
__device__ __forceinline__ void blur_vertical(const float (*hz)[SHL][HPITCH], int c, int vs, float (&o)[NQ][VSEG]) {
#pragma unroll
    for (int q = 0; q < NQ; ++q)
#pragma unroll
        for (int i = 0; i < VSEG; ++i) o[q][i] = 0.f;
#pragma unroll
    for (int k = 0; k < VSEG + 10; ++k) {
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const float v = hz[q][vs * VSEG + k][c];
#pragma unroll
            for (int i = 0; i < VSEG; ++i) {
                const int tap = k - i;
                if (tap >= 0 && tap <= 10) o[q][i] = __fmaf_rn(c_taps[tap], v, o[q][i]);
            }
        }
    }
}

__global__ void __launch_bounds__(LTHREADS) ssim_fwd_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                            int H, int W, float* __restrict__ map_mu,
                                                            float* __restrict__ map_s1, float* __restrict__ map_s12,
                                                            LossHdr* __restrict__ hdr, const float* __restrict__ depth,
                                                            const float* __restrict__ gt_depth, const float* __restrict__ alpha,
                                                            const int4* __restrict__ boxes, int n_boxes, LocalBox* __restrict__ lbox) {
    __shared__ float in[2][SHL][IPITCH];
    __shared__ float hz[5][SHL][HPITCH];
    __shared__ double red[8][LTHREADS / 32];
    __shared__ int near_box[LOCAL_BOXES_MAX];
    __shared__ int n_near_s;
    const int ch = blockIdx.z;
    const size_t plane = (size_t)ch * H * W;
    const int x0 = blockIdx.x * ST - HALO, y0 = blockIdx.y * ST - HALO;
    const bool local_boxes = ch == 0 && depth && n_boxes > 0;
    if (local_boxes && threadIdx.x < 32) {                 // (published by the barriers below)
        const int cnt = boxes_near_tile(boxes, n_boxes, blockIdx.x * ST, blockIdx.y * ST, near_box);
        if (threadIdx.x == 0) n_near_s = cnt;
    }
    for (int idx = threadIdx.x; idx < SHL * SHL; idx += LTHREADS) {
        const int r = idx / SHL, c = idx % SHL;
        const int y = y0 + r, x = x0 + c;
        float a = 0.f, b = 0.f;
        if (x >= 0 && x < W && y >= 0 && y < H) { a = pred[plane + (size_t)y * W + x]; b = gt[plane + (size_t)y * W + x]; }
        in[0][r][c] = a;
        in[1][r][c] = b;
    }
    __syncthreads();
    if (threadIdx.x < SHL * (ST / SEG)) {
        const int r = threadIdx.x % SHL, s = threadIdx.x / SHL;
        float a[5][SEG];
#pragma unroll
        for (int q = 0; q < 5; ++q)
#pragma unroll
            for (int i = 0; i < SEG; ++i) a[q][i] = 0.f;
#pragma unroll
        for (int k = 0; k < SEG + 10; ++k) {
            const float xv = in[0][r][s * SEG + k], yv = in[1][r][s * SEG + k];
            const float xx = xv * xv, yy = yv * yv, xy = xv * yv;
#pragma unroll
            for (int i = 0; i < SEG; ++i) {
                const int tap = k - i;
                if (tap >= 0 && tap <= 10) {
                    const float w = c_taps[tap];
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
            for (int i = 0; i < SEG; ++i) hz[q][r][s * SEG + i] = a[q][i];
    }
    __syncthreads();
    const int c = threadIdx.x % ST, vs = threadIdx.x / ST;
    float o[5][VSEG];
    blur_vertical<5>(hz, c, vs, o);
    const int x = blockIdx.x * ST + c;
    float ssim_v = 0.f, l1_v = 0.f;
    double st[6] = {0, 0, 0, 0, 0, 0};
    float dp[VSEG], dg[VSEG];                                     // this thread's depth pixels (channel-0 CTAs)
#pragma unroll
    for (int i = 0; i < VSEG; ++i) dp[i] = dg[i] = 0.f;
#pragma unroll
    for (int i = 0; i < VSEG; ++i) {
        const int y = blockIdx.y * ST + vs * VSEG + i;
        if (x < W && y < H) {
            const float mu1 = o[0][i], mu2 = o[1][i];
            const float mu1_sq = mu1 * mu1, mu2_sq = mu2 * mu2, mu12 = mu1 * mu2;
            const float s1 = o[2][i] - mu1_sq, s2 = o[3][i] - mu2_sq, s12 = o[4][i] - mu12;
            const float C1 = 0.0001f, C2 = 0.0009f;
            const float A1 = 2.f * mu12 + C1, A2 = 2.f * s12 + C2, B1 = mu1_sq + mu2_sq + C1, B2 = s1 + s2 + C2;
            const float inv = 1.0f / (B1 * B2);
            ssim_v += A1 * A2 * inv;
            const size_t hwpix = (size_t)y * W + x;
            if (map_mu) {
                // partial derivatives of the map w.r.t. (mu1 | E[x^2] | E[xy]) held independent
                const float d_s1 = -A1 * A2 * inv / B2;
                const float d_s12 = 2.f * A1 * inv;
                const float d_mu = (2.f * mu2 * B1 - A1 * 2.f * mu1) / (B1 * B1) * (A2 / B2) + d_s1 * (-2.f * mu1) + d_s12 * (-mu2);
                map_mu[plane + hwpix] = d_mu;
                map_s1[plane + hwpix] = d_s1;
                map_s12[plane + hwpix] = d_s12;
            }
            const int r = vs * VSEG + i + HALO;
            l1_v += fabsf(in[0][r][c + HALO] - in[1][r][c + HALO]);
            if (ch == 0) {
                if (depth) {
                    dp[i] = depth[hwpix]; dg[i] = gt_depth[hwpix];
                    const double p = dp[i], g = dg[i];
                    st[0] += p; st[1] += g; st[2] += p * p; st[3] += g * g; st[4] += p * g;
                }
                if (alpha) st[5] += (double)(1.0f - alpha[hwpix]);
            }
        }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    ssim_v = warp_sum(ssim_v);
    l1_v = warp_sum(l1_v);
    if (lane == 0) { red[0][warp] = ssim_v; red[1][warp] = l1_v; }
    const bool extras = ch == 0 && (depth || alpha);
    if (extras) {
#pragma unroll
        for (int k = 0; k < 6; ++k) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) st[k] += __shfl_xor_sync(0xffffffffu, st[k], off);
            if (lane == 0) red[2 + k][warp] = st[k];
        }
    }
    __syncthreads();
    if (threadIdx.x < (extras ? 8 : 2)) {
        double t = 0;
        for (int w = 0; w < LTHREADS / 32; ++w) t += red[threadIdx.x][w];
        atomicAdd(&hdr->sums[threadIdx.x], t);
    }
    // local Pearson boxes that overlap this tile (uniform loop; a 128x128 box overlaps ~1 % of the 32x32 tiles)
    if (local_boxes) {
        const int n_near = n_near_s;
        for (int kb = 0; kb < n_near; ++kb) {
            const int b = near_box[kb];
            const int4 bx = boxes[b];                             // row0, col0, rows, cols
            double s5[5] = {0, 0, 0, 0, 0};
            const bool xin = x >= bx.y && x < bx.y + bx.w && x < W;
#pragma unroll
            for (int i = 0; i < VSEG; ++i) {
                const int y = blockIdx.y * ST + vs * VSEG + i;
                if (xin && y >= bx.x && y < bx.x + bx.z && y < H) {
                    const double p = dp[i], g = dg[i];
                    s5[0] += p; s5[1] += g; s5[2] += p * p; s5[3] += g * g; s5[4] += p * g;
                }
            }
#pragma unroll
            for (int k = 0; k < 5; ++k) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) s5[k] += __shfl_xor_sync(0xffffffffu, s5[k], off);
                if (lane == 0 && s5[k] != 0.0) atomicAdd(&lbox[b].st[k], s5[k]);
            }
        }
    }
}

__global__ void __launch_bounds__(LTHREADS) ssim_bwd_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                            int H, int W, const float* __restrict__ map_mu,
                                                            const float* __restrict__ map_s1, const float* __restrict__ map_s12,
                                                            float k_ssim, float k_l1, float* __restrict__ dL_dpred,
                                                            const LossHdr* __restrict__ hdr, const float* __restrict__ depth,
                                                            const float* __restrict__ gt_depth, float* __restrict__ dL_ddepth,
                                                            float* __restrict__ dL_dalpha, const int4* __restrict__ boxes, int n_boxes,
                                                            const LocalBox* __restrict__ lbox) {
    __shared__ float in[3][SHL][IPITCH];
    __shared__ float hz[3][SHL][HPITCH];
    const int ch = blockIdx.z;
    const size_t plane = (size_t)ch * H * W;
    const int x0 = blockIdx.x * ST - HALO, y0 = blockIdx.y * ST - HALO;
    for (int idx = threadIdx.x; idx < SHL * SHL; idx += LTHREADS) {
        const int r = idx / SHL, c = idx % SHL;
        const int y = y0 + r, x = x0 + c;
        float a = 0.f, b = 0.f, d = 0.f;
        if (x >= 0 && x < W && y >= 0 && y < H) {
            const size_t pix = plane + (size_t)y * W + x;
            a = map_mu[pix]; b = map_s1[pix]; d = map_s12[pix];
        }
        in[0][r][c] = a; in[1][r][c] = b; in[2][r][c] = d;
    }
    __syncthreads();
    if (threadIdx.x < SHL * (ST / SEG)) {
        const int r = threadIdx.x % SHL, s = threadIdx.x / SHL;
        float a[3][SEG];
#pragma unroll
        for (int q = 0; q < 3; ++q)
#pragma unroll
            for (int i = 0; i < SEG; ++i) a[q][i] = 0.f;
#pragma unroll
        for (int k = 0; k < SEG + 10; ++k) {
            const float v0 = in[0][r][s * SEG + k], v1 = in[1][r][s * SEG + k], v2 = in[2][r][s * SEG + k];
#pragma unroll
            for (int i = 0; i < SEG; ++i) {
                const int tap = k - i;
                if (tap >= 0 && tap <= 10) {
                    const float w = c_taps[tap];
                    a[0][i] = __fmaf_rn(w, v0, a[0][i]);
                    a[1][i] = __fmaf_rn(w, v1, a[1][i]);
                    a[2][i] = __fmaf_rn(w, v2, a[2][i]);
                }
            }
        }
#pragma unroll
        for (int q = 0; q < 3; ++q)
#pragma unroll
            for (int i = 0; i < SEG; ++i) hz[q][r][s * SEG + i] = a[q][i];
    }
    __syncthreads();
    const int c = threadIdx.x % ST, vs = threadIdx.x / ST;
    float o[3][VSEG];
    blur_vertical<3>(hz, c, vs, o);
    const int x = blockIdx.x * ST + c;
    const bool do_depth = ch == 0 && dL_ddepth != nullptr, do_alpha = ch == 0 && dL_dalpha != nullptr;
    // the local boxes that overlap this tile, in box order (warp 0, ballot compaction: the per-pixel sum keeps one order)
    __shared__ int near_box[LOCAL_BOXES_MAX];
    __shared__ int n_near_s;
    if (do_depth && n_boxes > 0) {
        if (threadIdx.x < 32) {
            const int cnt = boxes_near_tile(boxes, n_boxes, blockIdx.x * ST, blockIdx.y * ST, near_box);
            if (threadIdx.x == 0) n_near_s = cnt;
        }
        __syncthreads();
    }
    const int n_near = (do_depth && n_boxes > 0) ? n_near_s : 0;
    float mg = 0.f, mp = 0.f, cg = 0.f, cp = 0.f, c0g = 0.f, ca = 0.f;
    if (do_depth) { mg = hdr->coef[0]; mp = hdr->coef[1]; cg = hdr->coef[2]; cp = hdr->coef[3]; c0g = hdr->coef[5]; }
    if (do_alpha) ca = hdr->coef[4];
#pragma unroll
    for (int i = 0; i < VSEG; ++i) {
        const int y = blockIdx.y * ST + vs * VSEG + i;
        if (x < W && y < H) {
            const size_t hwpix = (size_t)y * W + x, pix = plane + hwpix;
            const float xv = pred[pix], yv = gt[pix];
            const float dssim = o[0][i] + 2.f * xv * o[1][i] + yv * o[2][i];
            const float diff = xv - yv;
            const float sgn = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
            dL_dpred[pix] = k_ssim * dssim + k_l1 * sgn;
            if (do_depth) {
                const float g = gt_depth[hwpix], pv = depth[hwpix];
                float acc = cg * (g - mg) + cp * (pv - mp) + c0g;
                for (int k = 0; k < n_near; ++k) {                // every local box that covers this pixel adds its term
                    const int b = near_box[k];
                    const int4 bx = boxes[b];
                    if (y >= bx.x && y < bx.x + bx.z && x >= bx.y && x < bx.y + bx.w) {
                        const float4 c4 = *reinterpret_cast<const float4*>(lbox[b].coef);
                        acc += c4.z * (g - c4.x) + c4.w * (pv - c4.y) + lbox[b].c0;
                    }
                }
                dL_ddepth[hwpix] = acc;
            }
            if (do_alpha) dL_dalpha[hwpix] = ca;
        }
    }
}

// sums -> losses (+ the coefficients of the Pearson / alpha gradients for the second pass)
__global__ void loss_finalize_kernel(LossHdr* __restrict__ hdr, double n, double npix, float w_l1, float w_dssim,
                                     int use_depth, float w_pearson, float eps, int use_alpha, float w_alpha,
                                     float* __restrict__ out) {
    const double* sums = hdr->sums;
    const double ssim = sums[0] / n, l1 = sums[1] / n;
    out[0] = (float)(w_l1 * l1 + w_dssim * (1.0 - ssim));
    out[1] = (float)l1;
    out[2] = (float)ssim;
    if (use_depth) {
        // loss_utils.py:100-117: 1 - mean(z_p * z_g), z = (v - mean) / (std_unbiased + eps)
        const double m = npix;
        const double mp = sums[2] / m, mg = sums[3] / m;
        const double varp = fmax((sums[4] - m * mp * mp) / (m - 1.0), 0.0), varg = fmax((sums[5] - m * mg * mg) / (m - 1.0), 0.0);
        const double sp = sqrt(varp), sg = sqrt(varg);
        const double a = sp + (double)eps, b = sg + (double)eps;
        const double spg = sums[6] - m * mp * mg;
        out[3] = (float)(1.0 - spg / (m * a * b));
        const double k1 = 1.0 / (m * a * b);
        const double k2 = sp > 0.0 ? spg / (m * a * a * b) / ((m - 1.0) * sp) : 0.0;
        hdr->coef[0] = (float)mg;
        hdr->coef[1] = (float)mp;
        hdr->coef[2] = (float)(-(double)w_pearson * k1);
        hdr->coef[3] = (float)((double)w_pearson * k2);
        hdr->coef[5] = pearson_coef_correction(-(double)w_pearson * k1, mg, (double)w_pearson * k2, mp);
    }
    if (use_alpha) {
        out[4] = (float)((double)w_alpha * sums[7] / npix);
        hdr->coef[4] = (float)(-(double)w_alpha / npix);
    }
}

// LocalPearsonDepthLoss (losses.py:132-182): loss = mean_b (1 - Pearson_b); one thread per box
__global__ void local_pearson_finalize_kernel(LossHdr* __restrict__ hdr, const int4* __restrict__ boxes, int n_boxes,
                                              LocalBox* __restrict__ lbox, float w_local, float eps, float* __restrict__ out) {
    __shared__ double part[LOCAL_BOXES_MAX];
    const int b = threadIdx.x;
    double loss_b = 0.0;
    if (b < n_boxes) {
        const int4 bx = boxes[b];
        const double m = (double)bx.z * (double)bx.w;
        const double* st = lbox[b].st;
        const double mp = st[0] / m, mg = st[1] / m;
        const double varp = fmax((st[2] - m * mp * mp) / (m - 1.0), 0.0), varg = fmax((st[3] - m * mg * mg) / (m - 1.0), 0.0);
        const double sp = sqrt(varp), sg = sqrt(varg);
        const double a = sp + (double)eps, bb = sg + (double)eps;
        const double spg = st[4] - m * mp * mg;
        loss_b = 1.0 - spg / (m * a * bb);
        const double wgt = (double)w_local / (double)n_boxes;
        const double k1 = 1.0 / (m * a * bb);
        const double k2 = sp > 0.0 ? spg / (m * a * a * bb) / ((m - 1.0) * sp) : 0.0;
        lbox[b].coef[0] = (float)mg;
        lbox[b].coef[1] = (float)mp;
        lbox[b].coef[2] = (float)(-wgt * k1);
        lbox[b].coef[3] = (float)(wgt * k2);
        lbox[b].c0 = pearson_coef_correction(-wgt * k1, mg, wgt * k2, mp);
    }
    part[threadIdx.x] = loss_b;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < n_boxes; ++k) t += part[k];           // fixed order: reproducible
        out[5] = (float)(t / (double)n_boxes);
    }
}

// Workspace: LossHdr (256 B), the three derivative maps, then the LocalBox array.  The maps are rounded up to 256 B so that
// the boxes stay 16-byte aligned (pass 2 reads their coefficients as one float4) when C * H * W is not a multiple of 4.
static int64_t loss_boxes_offset(int64_t plane) { return 256 + rdg_align_up(3 * plane * (int64_t)sizeof(float), 256); }

extern "C" int64_t rdg_l1_dssim_workspace_bytes(int32_t channels, int32_t height, int32_t width) {
    if (channels <= 0 || height <= 0 || width <= 0) return RDG_E_ARG;
    return loss_boxes_offset((int64_t)channels * height * width) + (int64_t)LOCAL_BOXES_MAX * (int64_t)sizeof(LocalBox);
}

extern "C" int rdg_losses(const float* pred, const float* gt, int32_t channels, int32_t height, int32_t width,
                          float w_l1, float w_dssim, const RdgLossTerms* extra, float* out_loss, float* dL_dpred,
                          void* workspace, int64_t workspace_bytes, void* stream) {
    RDG_CHECK_ARG(pred && gt && out_loss && workspace, "null argument");
    RDG_CHECK_ARG(channels > 0 && height > 0 && width > 0, "empty image");
    if (workspace_bytes < rdg_l1_dssim_workspace_bytes(channels, height, width)) {
        rdg_set_error("rdg_losses: workspace too small");
        return RDG_E_CAPACITY;
    }
    const bool use_depth = extra && extra->depth && extra->gt_depth && extra->w_pearson != 0.0f;
    const bool use_alpha = extra && extra->alpha && extra->w_alpha != 0.0f;
    const bool use_local = extra && extra->depth && extra->gt_depth && extra->local_boxes && extra->n_local_boxes > 0 &&
                           extra->w_local != 0.0f;
    RDG_CHECK_ARG(!use_local || extra->n_local_boxes <= LOCAL_BOXES_MAX, "at most 256 local Pearson boxes");
    RDG_CHECK_ARG(!(use_local && dL_dpred) || extra->dL_ddepth, "the local Pearson term needs dL_ddepth");
    RDG_CHECK_ARG(((uintptr_t)workspace & 15) == 0, "workspace must be 16-byte aligned");
    const bool any_depth = use_depth || use_local;
    cudaStream_t s = (cudaStream_t)stream;
    LossHdr* hdr = (LossHdr*)workspace;
    const size_t plane = (size_t)channels * height * width;
    float* maps = (float*)((char*)workspace + 256);
    LocalBox* lbox = (LocalBox*)((char*)workspace + loss_boxes_offset((int64_t)plane));
    const int4* boxes = use_local ? (const int4*)extra->local_boxes : nullptr;
    const int n_boxes = use_local ? extra->n_local_boxes : 0;
    RDG_CUDA(cudaMemsetAsync(hdr, 0, sizeof(LossHdr), s));
    if (use_local) RDG_CUDA(cudaMemsetAsync(lbox, 0, (size_t)n_boxes * sizeof(LocalBox), s));
    const dim3 grid((width + ST - 1) / ST, (height + ST - 1) / ST, channels);
    const bool need_grad = dL_dpred != nullptr;
    ssim_fwd_kernel<<<grid, LTHREADS, 0, s>>>(pred, gt, height, width, need_grad ? maps : nullptr,
                                             need_grad ? maps + plane : nullptr, need_grad ? maps + 2 * plane : nullptr, hdr,
                                             any_depth ? extra->depth : nullptr, any_depth ? extra->gt_depth : nullptr,
                                             use_alpha ? extra->alpha : nullptr, boxes, n_boxes, lbox);
    RDG_CHECK_LAUNCH();
    const double n = (double)plane, npix = (double)height * (double)width;
    loss_finalize_kernel<<<1, 1, 0, s>>>(hdr, n, npix, w_l1, w_dssim, use_depth ? 1 : 0, use_depth ? extra->w_pearson : 0.f,
                                         use_depth ? extra->pearson_eps : 0.f, use_alpha ? 1 : 0,
                                         use_alpha ? extra->w_alpha : 0.f, out_loss);
    if (use_local)
        local_pearson_finalize_kernel<<<1, LOCAL_BOXES_MAX, 0, s>>>(hdr, boxes, n_boxes, lbox, extra->w_local, extra->pearson_eps, out_loss);
    if (need_grad) {
        ssim_bwd_kernel<<<grid, LTHREADS, 0, s>>>(pred, gt, height, width, maps, maps + plane, maps + 2 * plane,
                                                 (float)(-(double)w_dssim / n), (float)((double)w_l1 / n), dL_dpred, hdr,
                                                 any_depth ? extra->depth : nullptr, any_depth ? extra->gt_depth : nullptr,
                                                 any_depth ? extra->dL_ddepth : nullptr, use_alpha ? extra->dL_dalpha : nullptr,
                                                 boxes, n_boxes, lbox);
    }
    RDG_CHECK_LAUNCH();
    rdg_count_launches((need_grad ? 3 : 2) + (use_local ? 1 : 0));
    return RDG_OK;
}

extern "C" int rdg_l1_dssim(const float* pred, const float* gt, int32_t channels, int32_t height, int32_t width,
                            float w_l1, float w_dssim, float* out_loss, float* dL_dpred,
                            void* workspace, int64_t workspace_bytes, void* stream) {
    return rdg_losses(pred, gt, channels, height, width, w_l1, w_dssim, nullptr, out_loss, dL_dpred, workspace,
                      workspace_bytes, stream);
}

// ------------------------------------------------------------------ Pearson ----
// stats[b][0..4] = sum p, sum g, sum pp, sum gg, sum pg
__global__ void __launch_bounds__(RDG_BLOCK) pearson_stats_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                                  int W, const int4* __restrict__ boxes, double* __restrict__ stats) {
    __shared__ double red[5][RDG_BLOCK / 32];
    const int4 bx = boxes[blockIdx.y];   // row0, col0, rows, cols
    const int64_t n = (int64_t)bx.z * bx.w;
    double s[5] = {0, 0, 0, 0, 0};
    for (int64_t e = (int64_t)blockIdx.x * RDG_BLOCK + threadIdx.x; e < n; e += (int64_t)gridDim.x * RDG_BLOCK) {
        const int r = (int)(e / bx.w), c = (int)(e % bx.w);
        const size_t pix = (size_t)(bx.x + r) * W + bx.y + c;
        const double p = pred[pix], g = gt[pix];
        s[0] += p; s[1] += g; s[2] += p * p; s[3] += g * g; s[4] += p * g;
    }
#pragma unroll
    for (int k = 0; k < 5; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
        if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = s[k];
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        double t = 0;
        for (int w = 0; w < RDG_BLOCK / 32; ++w) t += red[threadIdx.x][w];
        atomicAdd(&stats[blockIdx.y * 8 + threadIdx.x], t);
    }
}

__global__ void __launch_bounds__(RDG_BLOCK) pearson_grad_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                                 int W, const int4* __restrict__ boxes, const float* __restrict__ box_weight,
                                                                 const double* __restrict__ stats, float eps,
                                                                 float* __restrict__ out_loss, float* __restrict__ dL_dpred) {
    const int4 bx = boxes[blockIdx.y];
    const double n = (double)bx.z * (double)bx.w;
    const double* st = stats + blockIdx.y * 8;
    const double mp = st[0] / n, mg = st[1] / n;
    const double varp = fmax((st[2] - n * mp * mp) / (n - 1.0), 0.0), varg = fmax((st[3] - n * mg * mg) / (n - 1.0), 0.0);
    const double sp = sqrt(varp), sg = sqrt(varg);
    const double a = sp + (double)eps, b = sg + (double)eps;
    const double spg = st[4] - n * mp * mg;
    const double cov = spg / (n * a * b);
    if (blockIdx.x == 0 && threadIdx.x == 0) out_loss[blockIdx.y] = (float)(1.0 - cov);
    if (!dL_dpred) return;
    const double wgt = box_weight ? (double)box_weight[blockIdx.y] : 1.0;
    const double k1 = 1.0 / (n * a * b);
    const double k2 = sp > 0.0 ? spg / (n * a * a * b) / ((n - 1.0) * sp) : 0.0;
    const int64_t cnt = (int64_t)bx.z * bx.w;
    for (int64_t e = (int64_t)blockIdx.x * RDG_BLOCK + threadIdx.x; e < cnt; e += (int64_t)gridDim.x * RDG_BLOCK) {
        const int r = (int)(e / bx.w), c = (int)(e % bx.w);
        const size_t pix = (size_t)(bx.x + r) * W + bx.y + c;
        const double p = pred[pix], g = gt[pix];
        const double dcov = (g - mg) * k1 - (p - mp) * k2;
        atomicAdd(&dL_dpred[pix], (float)(-wgt * dcov));
    }
}

extern "C" int rdg_pearson(const float* pred, const float* gt, int32_t height, int32_t width,
                           const int32_t* boxes, const float* box_weight, int32_t n_boxes, float eps,
                           float* out_loss, float* dL_dpred, double* stats, void* stream) {
    RDG_CHECK_ARG(pred && gt && boxes && out_loss && stats, "null argument");
    RDG_CHECK_ARG(height > 0 && width > 0, "empty image");
    if (n_boxes <= 0) return RDG_OK;
    cudaStream_t s = (cudaStream_t)stream;
    RDG_CUDA(cudaMemsetAsync(stats, 0, (size_t)n_boxes * 8 * sizeof(double), s));
    // whole-image boxes get many CTAs, 128x128 boxes a few
    const int per_box = n_boxes == 1 ? RDG_SM_COUNT * 2 : 8;
    const dim3 grid(per_box, n_boxes);
    pearson_stats_kernel<<<grid, RDG_BLOCK, 0, s>>>(pred, gt, width, (const int4*)boxes, stats);
    pearson_grad_kernel<<<grid, RDG_BLOCK, 0, s>>>(pred, gt, width, (const int4*)boxes, box_weight, stats, eps, out_loss, dL_dpred);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(2);
    return RDG_OK;
}

// ------------------------------------------------------------ alpha regulariser ----
__global__ void __launch_bounds__(RDG_BLOCK) alpha_reg_kernel(const float* __restrict__ alpha, int64_t n, float w_over_n,
                                                              float* __restrict__ out_loss, float* __restrict__ dL_dalpha) {
    __shared__ float red[RDG_BLOCK / 32];
    float s = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * RDG_BLOCK + threadIdx.x; i < n; i += (int64_t)gridDim.x * RDG_BLOCK) {
        s += 1.0f - alpha[i];
        if (dL_dalpha) dL_dalpha[i] = -w_over_n;
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int k = 0; k < RDG_BLOCK / 32; ++k) t += red[k];
        atomicAdd(out_loss, t * w_over_n);
    }
}

extern "C" int rdg_alpha_reg(const float* alpha, int64_t n, float weight, float* out_loss, float* dL_dalpha, void* stream) {
    RDG_CHECK_ARG(alpha && out_loss, "null argument");
    if (n <= 0) return RDG_OK;
    const int64_t want = (n + RDG_BLOCK - 1) / RDG_BLOCK;
    const int grid = (int)(want < (int64_t)RDG_SM_COUNT * 4 ? want : (int64_t)RDG_SM_COUNT * 4);
    alpha_reg_kernel<<<grid, RDG_BLOCK, 0, (cudaStream_t)stream>>>(alpha, n, weight / (float)n, out_loss, dL_dalpha);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}

// --------------------------------------------------------------------- Adam ----
__global__ void __launch_bounds__(RDG_BLOCK) adam_kernel(float* __restrict__ param, const float* __restrict__ grad,
                                                         float* __restrict__ m, float* __restrict__ v, int64_t n, float lr,
                                                         float b1, float b2, float eps, float bc1, float bc2_sqrt, float gscale) {
    for (int64_t i = (int64_t)blockIdx.x * RDG_BLOCK + threadIdx.x; i < n; i += (int64_t)gridDim.x * RDG_BLOCK) {
        const float g = grad[i] * gscale;
        const float mi = b1 * m[i] + (1.f - b1) * g;
        const float vi = b2 * v[i] + (1.f - b2) * g * g;
        m[i] = mi; v[i] = vi;
        // torch.optim.Adam: denom = sqrt(v)/sqrt(bias2) + eps; step = lr / bias1
        const float denom = sqrtf(vi) / bc2_sqrt + eps;
        param[i] -= (lr / bc1) * (mi / denom);
    }
}

extern "C" int rdg_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                        float lr, float beta1, float beta2, float eps, int32_t step, float grad_scale, void* stream) {
    RDG_CHECK_ARG(param && grad && exp_avg && exp_avg_sq, "null argument");
    RDG_CHECK_ARG(step >= 1, "step must be >= 1");
    if (n <= 0) return RDG_OK;
    const float bc1 = 1.0f - (float)pow((double)beta1, (double)step);
    const float bc2 = 1.0f - (float)pow((double)beta2, (double)step);
    const int64_t want = (n + RDG_BLOCK - 1) / RDG_BLOCK;
    const int grid = (int)(want < (int64_t)RDG_SM_COUNT * 8 ? want : (int64_t)RDG_SM_COUNT * 8);
    adam_kernel<<<grid, RDG_BLOCK, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps,
                                                            bc1, sqrtf(bc2), grad_scale);
    RDG_CHECK_LAUNCH();
    rdg_count_launches(1);
    return RDG_OK;
}
