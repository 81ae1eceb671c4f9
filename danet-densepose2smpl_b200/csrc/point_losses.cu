// Sparse losses of the training step, forward and backward in one pass each.
//
// DensePose points: models/danet/iuv_estimator.py:343-419 (IUV_Estimator.dp_uvia_losses) behind the has_dp selection of
// iuv_estimator.py:106-121, and the autograd graph torch builds for it (3 x grid_sample, 2 x cross-entropy, 2 x smooth-L1).
//   k_dp_points   one thread per (sample, point): bilinear corners, the 3C interpolated values, the point's loss terms
//                 and its gradient coefficients d loss / d interpolated value (workspace, [B][3C][P]).
//   k_dp_ann      one thread per (sample, pixel): cross-entropy of the annotation logits and its gradient (dense).
//   k_dp_scatter  the adjoint of the bilinear gather.  One CTA per (sample, channel group) counting-sorts the sample's
//                 4P (pixel, point, corner) entries by pixel in shared memory -- stable: entries keep point order --
//                 then every thread sums its pixel's entries in that order and writes the pixel (zero if untouched).
//   k_dp_finish   one block adds the per-point and per-block partials in double, in a fixed order.
// No float atomics anywhere (the counting sort uses integer ones): the result is bit-for-bit repeatable.
//
// STN key points: iuv_estimator.py:137-140 (soft-argmax centres, utils/keypoints.py:334-394) and :159-171 (loss_roi).
//   k_stn_kps     one CTA per (sample, joint): max, sum-exp and the two weighted sums of the S x S map, the centre, the
//                 joint's loss term and d loss / d map.
//   k_stn_finish  one block adds the joint terms in double, in a fixed order.
#include <algorithm>

#include "common.cuh"

namespace danet {

#ifdef __CUDA_ARCH__
#define DANET_PL_LDG(p) __ldg(p)
#else
#define DANET_PL_LDG(p) (*(p))
#endif

struct DpArgs {
    int B, C, Cann, S, P;
    const float *u, *v, *idx, *ann;           // [B,C,S,S] x 3, [B,Cann,S,S]
    const float *X, *Y, *I;                   // [B,P]
    const float *Up, *Vp, *Wp;                // [B,C*P]: channel c of point p at c*P + p
    const float* alab;                        // [B,S*S]
    const uint8_t* has;                       // [B] or NULL
    int align;                                // grid_sample align_corners
    float iw, partw, pointw;                  // INDEX_WEIGHTS, PART_WEIGHTS, POINT_REGRESSION_WEIGHTS
    float *gu, *gv, *gidx, *gann;
    int4* pix;                                // [B][P]: corner pixels nw, ne, sw, se (-1: outside / sample not selected)
    float4* cw;                               // [B][P]: corner weights
    float* gpt;                               // [B][3C][P]: d loss / d interpolated u, v, index
    float4* ptl;                              // [B][P]: the point's loss terms (u, v, index), un-normalised
    float* apart;                             // k_dp_ann block partials
    float* losses;
};

__host__ __device__ inline float sl1(float d) { const float a = fabsf(d); return a < 1.f ? 0.5f * d * d : a - 0.5f; }
__host__ __device__ inline float clamp1(float d) { return fminf(fmaxf(d, -1.f), 1.f); }

// grid_sample's bilinear corners (zero padding) at point p of sample n, in the arithmetic of torch's CPU kernel:
// grid = (X - S/2) * (2/S) (iuv_estimator.py:387-389), un-normalised as (g + 1) * (S-1)/2 (align_corners) or as one
// fused (g + 1) * S/2 - 0.5, weights from the fractional parts.
__host__ __device__ inline void dp_corners(const DpArgs& a, int n, int p, int4& pix, float4& w) {
    const int S = a.S;
    const float half = (float)(0.5 * S), scale = (float)(2.0 / S);
    const float gx = (DANET_PL_LDG(a.X + (size_t)n * a.P + p) - half) * scale;
    const float gy = (DANET_PL_LDG(a.Y + (size_t)n * a.P + p) - half) * scale;
    float ix, iy;
    if (a.align) {
        const float f = (float)(S - 1) / 2.f;
        ix = (gx + 1.f) * f; iy = (gy + 1.f) * f;
    } else {
        const float f = (float)S / 2.f;
        ix = fmaf(gx + 1.f, f, -0.5f); iy = fmaf(gy + 1.f, f, -0.5f);
    }
    const float x0 = floorf(ix), y0 = floorf(iy);
    const float wx = ix - x0, ex = 1.f - wx, wy = iy - y0, ey = 1.f - wy;
    w = make_float4(ey * ex, ey * wx, wy * ex, wy * wx);
    const float Sf = (float)S;
    const bool x0in = x0 >= 0.f && x0 < Sf, x1in = x0 + 1.f >= 0.f && x0 + 1.f < Sf;
    const bool y0in = y0 >= 0.f && y0 < Sf, y1in = y0 + 1.f >= 0.f && y0 + 1.f < Sf;
    const int xi = (x0in || x1in) ? (int)x0 : 0, yi = (y0in || y1in) ? (int)y0 : 0;
    pix.x = (y0in && x0in) ? yi * S + xi : -1;
    pix.y = (y0in && x1in) ? yi * S + xi + 1 : -1;
    pix.z = (y1in && x0in) ? (yi + 1) * S + xi : -1;
    pix.w = (y1in && x1in) ? (yi + 1) * S + xi + 1 : -1;
}

// the interpolated value: nw first, then one fused multiply-add per further corner (torch's CPU order)
__host__ __device__ inline float bilinear(const float* __restrict__ m, int4 pix, float4 w) {
    const float a = pix.x >= 0 ? DANET_PL_LDG(m + pix.x) : 0.f, b = pix.y >= 0 ? DANET_PL_LDG(m + pix.y) : 0.f;
    const float c = pix.z >= 0 ? DANET_PL_LDG(m + pix.z) : 0.f, d = pix.w >= 0 ? DANET_PL_LDG(m + pix.w) : 0.f;
    return fmaf(d, w.w, fmaf(c, w.z, fmaf(b, w.y, a * w.x)));
}

// cross-entropy label: .to(torch.int64) truncates; a label outside [0, K) makes the loss NaN (the reference raises)
__host__ __device__ inline bool ce_label(float l, int K, int& t) {
    const bool ok = l > -1.f && l < (float)K;
    t = ok ? (int)l : 0;
    return ok;
}

// Everything point p of sample n contributes: the loss terms (u, v, index; un-normalised, returned) and the gradient
// coefficients g[k * gs], k < 3C (u channels, v channels, index channels).  inv_np = 1 / (selected samples * P).
// Shared by the kernel and by the host walk the CPU tests compile (DANET_POINT_LOSSES_HOST_CHECK).
__host__ __device__ inline float4 dp_point(const DpArgs& a, int n, int p, int4 pix, float4 w, float inv_np, float* g,
                                           size_t gs) {
    const int C = a.C, P = a.P;
    const size_t HW = (size_t)a.S * a.S;
    float l[2] = {0.f, 0.f};
    for (int k = 0; k < 2; ++k) {
        const float* m = (k == 0 ? a.u : a.v) + (size_t)n * C * HW;
        const float* t = (k == 0 ? a.Up : a.Vp) + (size_t)n * C * P + p;
        const float* pw = a.Wp + (size_t)n * C * P + p;
        for (int c = 0; c < C; ++c) {
            const float wt = DANET_PL_LDG(pw + (size_t)c * P);
            const float d = wt * (bilinear(m + c * HW, pix, w) - DANET_PL_LDG(t + (size_t)c * P));   // utils/net.py:18-35
            l[k] += wt * sl1(d);
            g[(size_t)(k * C + c) * gs] = a.pointw * wt * wt * clamp1(d);
        }
    }
    // cross-entropy of the interpolated index logits; the logits pass through g
    const float* m = a.idx + (size_t)n * C * HW;
    float* gi = g + (size_t)2 * C * gs;
    float mx = -INFINITY, s = 0.f;
    for (int c = 0; c < C; ++c) {
        const float x = bilinear(m + c * HW, pix, w);
        gi[(size_t)c * gs] = x;
        if (x > mx) { s = s * expf(mx - x) + 1.f; mx = x; } else s += expf(x - mx);
    }
    int t;
    const bool ok = ce_label(DANET_PL_LDG(a.I + (size_t)n * P + p), C, t);
    const float li = ok ? mx + logf(s) - gi[(size_t)t * gs] : NAN;
    const float sc = a.partw * inv_np, inv = 1.f / s;
    for (int c = 0; c < C; ++c) {
        const float x = gi[(size_t)c * gs];
        gi[(size_t)c * gs] = ok ? (expf(x - mx) * inv - (c == t ? 1.f : 0.f)) * sc : NAN;
    }
    return make_float4(l[0], l[1], li, 0.f);
}

// cross-entropy of the annotation logits at pixel q of sample n (iuv_estimator.py:399-404); writes d / d logits
// (scale = INDEX_WEIGHTS / (selected samples * S^2)) when a.gann is set, returns the un-normalised loss term
__host__ __device__ inline float dp_ann_pixel(const DpArgs& a, int n, int q, bool on, float scale) {
    const size_t HW = (size_t)a.S * a.S;
    const float* x = a.ann + (size_t)n * a.Cann * HW + q;
    float* g = a.gann ? a.gann + (size_t)n * a.Cann * HW + q : nullptr;
    if (!on) {
        if (g) for (int c = 0; c < a.Cann; ++c) g[c * HW] = 0.f;
        return 0.f;
    }
    int t;
    const bool ok = ce_label(DANET_PL_LDG(a.alab + (size_t)n * HW + q), a.Cann, t);
    float m = -INFINITY, s = 0.f, xt = 0.f;
    for (int c = 0; c < a.Cann; ++c) {
        const float xv = DANET_PL_LDG(x + c * HW);
        if (c == t) xt = xv;
        if (xv > m) { s = s * expf(m - xv) + 1.f; m = xv; } else s += expf(xv - m);
    }
    if (g) {
        const float inv = 1.f / s;
        for (int c = 0; c < a.Cann; ++c)
            g[c * HW] = ok ? (expf(DANET_PL_LDG(x + c * HW) - m) * inv - (c == t ? 1.f : 0.f)) * scale : NAN;
    }
    return ok ? m + logf(s) - xt : NAN;
}

// one gradient entry of the scatter: acc + corner weight * point coefficient, fused (kernel and host walk agree bitwise)
__host__ __device__ inline float scatter_add(float acc, float w, float g) { return fmaf(w, g, acc); }

// number of selected samples; every thread of the block must call it
__device__ inline int count_selected(const uint8_t* has, int B) {
    int c = 0;
    for (int base = 0; base < B; base += blockDim.x) {
        const int i = base + threadIdx.x;
        c += __syncthreads_count(i < B && (has == nullptr || has[i] != 0));
    }
    return c;
}

__global__ void __launch_bounds__(64) k_dp_points(const DpArgs a) {
    const int nsel = count_selected(a.has, a.B);
    const int n = blockIdx.y, p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.P) return;
    const size_t o = (size_t)n * a.P + p;
    int4 pix = make_int4(-1, -1, -1, -1);
    float4 w = make_float4(0.f, 0.f, 0.f, 0.f), l = w;
    if (a.has == nullptr || a.has[n] != 0) {
        dp_corners(a, n, p, pix, w);
        l = dp_point(a, n, p, pix, w, 1.f / ((float)nsel * (float)a.P), a.gpt + (size_t)n * 3 * a.C * a.P + p, a.P);
    }
    a.pix[o] = pix; a.cw[o] = w; a.ptl[o] = l;
}

__global__ void __launch_bounds__(256) k_dp_ann(const DpArgs a) {
    const int nsel = count_selected(a.has, a.B);
    const int HW = a.S * a.S;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    float l = 0.f;
    if (gid < (long long)a.B * HW) {
        const int n = (int)(gid / HW), q = (int)(gid - (long long)n * HW);
        const bool on = a.has == nullptr || a.has[n] != 0;
        l = dp_ann_pixel(a, n, q, on, on ? a.iw / ((float)nsel * (float)HW) : 0.f);
    }
    __shared__ float sm[8];
    l = warp_sum(l);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = l;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = sm[0];
        for (int i = 1; i < (int)(blockDim.x >> 5); ++i) t += sm[i];
        a.apart[blockIdx.x] = t;
    }
}

static inline size_t dp_scatter_smem(int S, int P) { return ((size_t)2 * S * S + 1 + (size_t)3 * 4 * P) * sizeof(int); }

// blockIdx.y = sample, blockIdx.x = group of `cpg` consecutive channels of the 3C (u, v, index) gradient planes
__global__ void __launch_bounds__(256) k_dp_scatter(const DpArgs a, int cpg) {
    extern __shared__ int sm[];
    const int n = blockIdx.y, HW = a.S * a.S, E = 4 * a.P, C = a.C;
    const int k0 = blockIdx.x * cpg, k1 = min(3 * C, k0 + cpg);
    float* planes[3] = {a.gu, a.gv, a.gidx};
    bool any = false;
    for (int k = k0; k < k1; ++k) any |= planes[k / C] != nullptr;
    if (!any) return;                                             // uniform across the block
    int* start = sm;                                              // [HW + 1] first sorted entry of each pixel
    int* cur = start + HW + 1;                                    // [HW] counts, then placement cursors
    int* order = cur + HW;                                        // [E] entry ids sorted by pixel, point order kept
    int* epix = order + E;                                        // [E]
    float* ew = reinterpret_cast<float*>(epix + E);               // [E]
    for (int q = threadIdx.x; q < HW; q += blockDim.x) cur[q] = 0;
    __syncthreads();
    const int* gpix = reinterpret_cast<const int*>(a.pix + (size_t)n * a.P);
    const float* gw = reinterpret_cast<const float*>(a.cw + (size_t)n * a.P);
    for (int e = threadIdx.x; e < E; e += blockDim.x) {
        const int q = gpix[e];
        epix[e] = q; ew[e] = gw[e];
        if (q >= 0) atomicAdd(&cur[q], 1);                        // integer: order-independent
    }
    __syncthreads();
    // exclusive scan of the counts: a contiguous chunk per thread, then the chunk totals across the block
    const int chunk = (HW + blockDim.x - 1) / blockDim.x, lo = min(HW, (int)threadIdx.x * chunk), hi = min(HW, lo + chunk);
    int tsum = 0;
    for (int q = lo; q < hi; ++q) tsum += cur[q];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = tsum;
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
    __shared__ int wtot[8];
    if (lane == 31) wtot[warp] = incl;
    __syncthreads();
    int run = incl - tsum;
    for (int i = 0; i < warp; ++i) run += wtot[i];
    for (int q = lo; q < hi; ++q) { const int c = cur[q]; start[q] = run; cur[q] = run; run += c; }
    if (threadIdx.x == blockDim.x - 1) start[HW] = run;
    __syncthreads();
    // stable placement by one warp, 32 entries at a time: the lanes that share a pixel take consecutive slots in lane
    // (= entry) order, and the highest of them advances the pixel's cursor
    if (warp == 0) {
        for (int base = 0; base < E; base += 32) {
            const int e = base + lane;
            const int q = e < E ? epix[e] : -1;
            const unsigned peers = __match_any_sync(0xffffffffu, q);
            if (q >= 0) order[cur[q] + __popc(peers & ((1u << lane) - 1u))] = e;
            __syncwarp();
            if (q >= 0 && lane == 31 - __clz(peers)) cur[q] += __popc(peers);
            __syncwarp();
        }
    }
    __syncthreads();
    for (int k = k0; k < k1; ++k) {
        float* out = planes[k / C];
        if (!out) continue;
        out += ((size_t)n * C + k % C) * HW;
        const float* g = a.gpt + ((size_t)n * 3 * C + k) * a.P;
        for (int q = threadIdx.x; q < HW; q += blockDim.x) {
            float acc = 0.f;
            for (int i = start[q]; i < start[q + 1]; ++i) {
                const int e = order[i];
                acc = scatter_add(acc, ew[e], __ldg(g + (e >> 2)));
            }
            out[q] = acc;
        }
    }
}

__device__ inline void block_sum_double(double* v, int nv, double (*sm)[256]) {
    for (int k = 0; k < nv; ++k) sm[k][threadIdx.x] = v[k];
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) for (int k = 0; k < nv; ++k) sm[k][threadIdx.x] += sm[k][threadIdx.x + o];
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) k_dp_finish(const DpArgs a, int ann_blocks) {
    const int nsel = count_selected(a.has, a.B);
    __shared__ double sm[4][256];
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < a.B * a.P; i += 256) { const float4 t = a.ptl[i]; s[0] += t.x; s[1] += t.y; s[2] += t.z; }
    for (int i = threadIdx.x; i < ann_blocks; i += 256) s[3] += a.apart[i];
    block_sum_double(s, 4, sm);
    if (threadIdx.x == 0) {
        const double np = (double)nsel * a.P, npix = (double)nsel * a.S * a.S;
        a.losses[0] = (float)(sm[0][0] * a.pointw);
        a.losses[1] = (float)(sm[1][0] * a.pointw);
        a.losses[2] = nsel > 0 ? (float)(sm[2][0] * a.partw / np) : 0.f;
        a.losses[3] = nsel > 0 ? (float)(sm[3][0] * a.iw / npix) : 0.f;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
struct StnArgs {
    int B, J, S;
    const float* hm;                          // [B,J,S,S]
    const float* kps;                         // [B,J,3]: x, y in [-1, 1], weight
    float weight;                             // STN_KPS_WEIGHTS
    float *centers, *ghm, *jl, *loss;         // [B,J,2], [B,J,S,S] or NULL, [B*J] joint terms, [1]
};

// joint bj from the softmax statistics of 10 * map (sum s, column- and row-weighted sums sx, sy): sets the raw
// integrals hat, the centre c (iuv_estimator.py:137-140) and gc = d loss_roi / d c; returns the joint's loss term
// w * sum_xy smooth_l1(c - gt)
__host__ __device__ inline float stn_joint(const StnArgs& a, int bj, float s, float sx, float sy, float2& hat, float2& c,
                                           float2& gc) {
    hat = make_float2(sx / s, sy / s);
    const float half = 0.5f * (float)a.S;
    const float cx = hat.x / half - 1.f, cy = hat.y / half - 1.f;
    c = make_float2(cx, cy);
    const float gx = DANET_PL_LDG(a.kps + 3 * bj), gy = DANET_PL_LDG(a.kps + 3 * bj + 1), w = DANET_PL_LDG(a.kps + 3 * bj + 2);
    gc = make_float2(0.f, 0.f);
    if (w == 0.f) return 0.f;                                     // iuv_estimator.py:164-165
    const float dx = cx - gx, dy = cy - gy, sc = a.weight * w / (float)a.B;
    gc = make_float2(clamp1(dx) * sc, clamp1(dy) * sc);
    return w * (sl1(dx) + sl1(dy));
}

// d loss_roi / d map at pixel (row, col): (10 / (S/2)) * softmax * (gc.x (col - x^) + gc.y (row - y^))
__host__ __device__ inline float stn_pixel_grad(const StnArgs& a, float e, float inv_s, int row, int col, float2 hat, float2 gc) {
    return (10.f / (0.5f * (float)a.S)) * (e * inv_s) * (gc.x * ((float)col - hat.x) + gc.y * ((float)row - hat.y));
}

__global__ void __launch_bounds__(256) k_stn_kps(const StnArgs a) {
    const int bj = blockIdx.x, S = a.S, HW = S * S;
    const float* x = a.hm + (size_t)bj * HW;
    __shared__ float sm[3][8];
    __shared__ float bc[3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    float m = -INFINITY;
    for (int p = threadIdx.x; p < HW; p += blockDim.x) m = fmaxf(m, 10.f * __ldg(x + p));
    m = warp_max(m);
    if (lane == 0) sm[0][warp] = m;
    __syncthreads();
    if (threadIdx.x == 0) { float t = sm[0][0]; for (int i = 1; i < nw; ++i) t = fmaxf(t, sm[0][i]); bc[0] = t; }
    __syncthreads();
    m = bc[0];
    float s = 0.f, sx = 0.f, sy = 0.f;
    for (int p = threadIdx.x; p < HW; p += blockDim.x) {
        const float e = expf(10.f * __ldg(x + p) - m);
        s += e; sx = fmaf(e, (float)(p % S), sx); sy = fmaf(e, (float)(p / S), sy);
    }
    s = warp_sum(s); sx = warp_sum(sx); sy = warp_sum(sy);
    __syncthreads();
    if (lane == 0) { sm[0][warp] = s; sm[1][warp] = sx; sm[2][warp] = sy; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float t0 = sm[0][0], t1 = sm[1][0], t2 = sm[2][0];
        for (int i = 1; i < nw; ++i) { t0 += sm[0][i]; t1 += sm[1][i]; t2 += sm[2][i]; }
        bc[0] = t0; bc[1] = t1; bc[2] = t2;
    }
    __syncthreads();
    float2 hat, c, gc;
    const float l = stn_joint(a, bj, bc[0], bc[1], bc[2], hat, c, gc);   // every thread: same inputs, same result
    if (threadIdx.x == 0) { a.jl[bj] = l; a.centers[2 * bj] = c.x; a.centers[2 * bj + 1] = c.y; }
    if (a.ghm) {
        const float inv = 1.f / bc[0];
        float* g = a.ghm + (size_t)bj * HW;
        for (int p = threadIdx.x; p < HW; p += blockDim.x)
            g[p] = stn_pixel_grad(a, expf(10.f * __ldg(x + p) - m), inv, p / S, p % S, hat, gc);
    }
}

__global__ void __launch_bounds__(256) k_stn_finish(const StnArgs a) {
    __shared__ double sm[1][256];
    double s = 0.0;
    for (int i = threadIdx.x; i < a.B * a.J; i += 256) s += a.jl[i];
    block_sum_double(&s, 1, sm);
    if (threadIdx.x == 0) a.loss[0] = a.B > 0 ? (float)(sm[0][0] * a.weight / a.B) : 0.f;
}

}  // namespace danet

using namespace danet;

namespace {
struct DpLayout { size_t pix, cw, gpt, ptl, apart, total; int ann_blocks; };
DpLayout dp_layout(long long B, long long C, long long S, long long P) {
    DpLayout L;
    const long long bp = B * P;
    L.ann_blocks = (int)((B * S * S + 255) / 256);
    L.pix = 0;
    L.cw = align_up(L.pix + bp * sizeof(int4), 256);
    L.gpt = align_up(L.cw + bp * sizeof(float4), 256);
    L.ptl = align_up(L.gpt + bp * 3 * C * sizeof(float), 256);
    L.apart = align_up(L.ptl + bp * sizeof(float4), 256);
    L.total = align_up(L.apart + (L.ann_blocks > 0 ? L.ann_blocks : 1) * sizeof(float), 256);
    return L;
}
}  // namespace

extern "C" int64_t danet_dp_uvia_losses_workspace_bytes(int32_t B, int32_t C, int32_t S, int32_t P) {
    if (B < 0 || C < 0 || S < 0 || P < 0) return -1;
    return (int64_t)dp_layout(B, C, S, P).total;
}

extern "C" int danet_dp_uvia_losses(int32_t B, int32_t C, int32_t Cann, int32_t S, int32_t P, const float* u_pred,
                                    const float* v_pred, const float* index_pred, const float* ann_pred,
                                    const float* X_points, const float* Y_points, const float* I_points,
                                    const float* U_points, const float* V_points, const float* point_weights,
                                    const float* ann_labels, const uint8_t* has_dp, int32_t align_corners,
                                    float index_weight, float part_weight, float point_weight, float* losses,
                                    float* grad_u, float* grad_v, float* grad_index, float* grad_ann, void* workspace,
                                    danet_stream_t stream) {
    DANET_CHECK(B >= 0 && C >= 1 && Cann >= 1 && S >= 1 && P >= 1, "dp_uvia_losses: bad sizes B=%d C=%d Cann=%d S=%d P=%d",
                B, C, Cann, S, P);
    DANET_CHECK(losses && workspace, "dp_uvia_losses: null pointer");
    DANET_CHECK(B == 0 || (u_pred && v_pred && index_pred && ann_pred && X_points && Y_points && I_points && U_points &&
                           V_points && point_weights && ann_labels), "dp_uvia_losses: null input pointer");
    const size_t smem = dp_scatter_smem(S, P);
    DANET_CHECK(smem <= 227 * 1024, "dp_uvia_losses: S=%d P=%d exceed the scatter's shared memory", S, P);
    DANET_CHECK((long long)B * S * S / 256 < (1LL << 31), "dp_uvia_losses: too many pixels");
    cudaStream_t st = (cudaStream_t)stream;
    const DpLayout L = dp_layout(B, C, S, P);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    DpArgs a;
    a.B = B; a.C = C; a.Cann = Cann; a.S = S; a.P = P;
    a.u = u_pred; a.v = v_pred; a.idx = index_pred; a.ann = ann_pred;
    a.X = X_points; a.Y = Y_points; a.I = I_points; a.Up = U_points; a.Vp = V_points; a.Wp = point_weights;
    a.alab = ann_labels; a.has = has_dp; a.align = align_corners ? 1 : 0;
    a.iw = index_weight; a.partw = part_weight; a.pointw = point_weight;
    a.gu = grad_u; a.gv = grad_v; a.gidx = grad_index; a.gann = grad_ann;
    a.pix = reinterpret_cast<int4*>(ws + L.pix); a.cw = reinterpret_cast<float4*>(ws + L.cw);
    a.gpt = reinterpret_cast<float*>(ws + L.gpt); a.ptl = reinterpret_cast<float4*>(ws + L.ptl);
    a.apart = reinterpret_cast<float*>(ws + L.apart); a.losses = losses;
    if (B > 0) {
        k_dp_points<<<dim3(cdiv(P, 64), B), 64, 0, st>>>(a);
        DANET_LAUNCH_CHECK();
        k_dp_ann<<<L.ann_blocks, 256, 0, st>>>(a);
        DANET_LAUNCH_CHECK();
        if (grad_u || grad_v || grad_index) {
            // enough CTAs to cover the SMs twice: each re-sorts its sample's entries (a few microseconds) and writes
            // cpg gradient planes
            const int groups = std::min(3 * C, std::max(1, cdiv(2 * 148, B)));
            const int cpg = cdiv(3 * C, groups);
            if (smem > 48 * 1024) DANET_CUDA(cudaFuncSetAttribute(k_dp_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_dp_scatter<<<dim3(cdiv(3 * C, cpg), B), 256, smem, st>>>(a, cpg);
            DANET_LAUNCH_CHECK();
        }
    }
    k_dp_finish<<<1, 256, 0, st>>>(a, B > 0 ? L.ann_blocks : 0);
    DANET_LAUNCH_CHECK();
    return 0;
}

extern "C" int64_t danet_stn_kps_losses_workspace_bytes(int32_t B, int32_t J) {
    if (B < 0 || J < 0) return -1;
    return align_up((int64_t)(B * (int64_t)J > 0 ? B * (int64_t)J : 1) * (int64_t)sizeof(float), 256);
}

extern "C" int danet_stn_kps_losses(int32_t B, int32_t J, int32_t S, const float* hm, const float* kps_gt, float weight,
                                    float* loss, float* centers, float* grad_hm, void* workspace, danet_stream_t stream) {
    DANET_CHECK(B >= 0 && J >= 1 && S >= 1, "stn_kps_losses: bad sizes B=%d J=%d S=%d", B, J, S);
    DANET_CHECK(loss && workspace && (B == 0 || (hm && kps_gt && centers)), "stn_kps_losses: null pointer");
    DANET_CHECK((long long)B * J < (1LL << 31), "stn_kps_losses: too many maps");
    cudaStream_t st = (cudaStream_t)stream;
    StnArgs a;
    a.B = B; a.J = J; a.S = S; a.hm = hm; a.kps = kps_gt; a.weight = weight;
    a.centers = centers; a.ghm = grad_hm; a.jl = reinterpret_cast<float*>(workspace); a.loss = loss;
    if (B > 0) {
        k_stn_kps<<<B * J, 256, 0, st>>>(a);
        DANET_LAUNCH_CHECK();
    }
    k_stn_finish<<<1, 256, 0, st>>>(a);
    DANET_LAUNCH_CHECK();
    return 0;
}

#ifdef DANET_POINT_LOSSES_HOST_CHECK
// Test-only (never part of libdanet_b200.so: the flag is set by tests/test_point_losses_cpu.py alone): the per-point,
// per-pixel and per-joint functions of the kernels walked on the host over HOST arrays, the scatter in the kernel's
// entry order, so that the arithmetic is pinned against the reference-generated golden without a GPU.
extern "C" int danet_test_dp_uvia_losses_host(int32_t B, int32_t C, int32_t Cann, int32_t S, int32_t P, const float* u,
                                              const float* v, const float* idx, const float* ann, const float* X,
                                              const float* Y, const float* I, const float* Up, const float* Vp,
                                              const float* Wp, const float* alab, const uint8_t* has, int32_t align,
                                              float iw, float partw, float pointw, float* losses, float* gu, float* gv,
                                              float* gidx, float* gann) {
    DpArgs a;
    a.B = B; a.C = C; a.Cann = Cann; a.S = S; a.P = P;
    a.u = u; a.v = v; a.idx = idx; a.ann = ann; a.X = X; a.Y = Y; a.I = I; a.Up = Up; a.Vp = Vp; a.Wp = Wp;
    a.alab = alab; a.has = has; a.align = align; a.iw = iw; a.partw = partw; a.pointw = pointw;
    a.gu = gu; a.gv = gv; a.gidx = gidx; a.gann = gann;
    int nsel = 0;
    for (int n = 0; n < B; ++n) nsel += (!has || has[n]) ? 1 : 0;
    const int HW = S * S;
    std::vector<int4> pix(P);
    std::vector<float4> cw(P);
    std::vector<float> gpt((size_t)3 * C * P);
    double s[4] = {0, 0, 0, 0};
    float* planes[3] = {gu, gv, gidx};
    for (int n = 0; n < B; ++n) {
        const bool on = !has || has[n];
        for (int p = 0; p < P; ++p) {
            pix[p] = make_int4(-1, -1, -1, -1);
            cw[p] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!on) continue;
            dp_corners(a, n, p, pix[p], cw[p]);
            const float4 l = dp_point(a, n, p, pix[p], cw[p], 1.f / ((float)nsel * (float)P), gpt.data() + p, P);
            s[0] += l.x; s[1] += l.y; s[2] += l.z;
        }
        for (int k = 0; k < 3 * C; ++k) {
            float* out = planes[k / C];
            if (!out) continue;
            out += ((size_t)n * C + k % C) * HW;
            std::vector<float> acc(HW, 0.f);
            for (int p = 0; p < P; ++p) {
                const int q[4] = {pix[p].x, pix[p].y, pix[p].z, pix[p].w};
                const float w[4] = {cw[p].x, cw[p].y, cw[p].z, cw[p].w};
                for (int c = 0; c < 4; ++c)
                    if (q[c] >= 0) acc[q[c]] = scatter_add(acc[q[c]], w[c], gpt[(size_t)k * P + p]);
            }
            for (int q = 0; q < HW; ++q) out[q] = acc[q];
        }
        for (int q = 0; q < HW; ++q) s[3] += dp_ann_pixel(a, n, q, on, on ? iw / ((float)nsel * (float)HW) : 0.f);
    }
    losses[0] = (float)(s[0] * pointw); losses[1] = (float)(s[1] * pointw);
    losses[2] = nsel > 0 ? (float)(s[2] * partw / ((double)nsel * P)) : 0.f;
    losses[3] = nsel > 0 ? (float)(s[3] * iw / ((double)nsel * HW)) : 0.f;
    return 0;
}

extern "C" int danet_test_stn_kps_losses_host(int32_t B, int32_t J, int32_t S, const float* hm, const float* kps, float weight,
                                              float* loss, float* centers, float* ghm) {
    StnArgs a;
    a.B = B; a.J = J; a.S = S; a.hm = hm; a.kps = kps; a.weight = weight; a.centers = centers; a.ghm = ghm;
    a.jl = nullptr; a.loss = loss;
    const int HW = S * S, T = 256;
    double tot = 0.0;
    for (int bj = 0; bj < B * J; ++bj) {
        const float* x = hm + (size_t)bj * HW;
        float m = -INFINITY;
        for (int p = 0; p < HW; ++p) m = fmaxf(m, 10.f * x[p]);
        // k_stn_kps's order: per-thread strided sums, xor-shuffle trees within the warps, then the warps in order
        float r[3][T];
        for (int t = 0; t < T; ++t) {
            float s = 0.f, sx = 0.f, sy = 0.f;
            for (int p = t; p < HW; p += T) {
                const float e = expf(10.f * x[p] - m);
                s += e; sx = fmaf(e, (float)(p % S), sx); sy = fmaf(e, (float)(p / S), sy);
            }
            r[0][t] = s; r[1][t] = sx; r[2][t] = sy;
        }
        float tsum[3] = {0.f, 0.f, 0.f};
        for (int k = 0; k < 3; ++k) {
            for (int w = 0; w < T / 32; ++w) {
                float* v = r[k] + 32 * w;
                for (int o = 16; o > 0; o >>= 1) {
                    float nv[32];
                    for (int l = 0; l < 32; ++l) nv[l] = v[l] + v[l ^ o];
                    for (int l = 0; l < 32; ++l) v[l] = nv[l];
                }
                tsum[k] = w == 0 ? v[0] : tsum[k] + v[0];
            }
        }
        const float s = tsum[0];
        float2 hat, c, gc;
        tot += stn_joint(a, bj, s, tsum[1], tsum[2], hat, c, gc);
        centers[2 * bj] = c.x; centers[2 * bj + 1] = c.y;
        if (ghm)
            for (int p = 0; p < HW; ++p) ghm[(size_t)bj * HW + p] = stn_pixel_grad(a, expf(10.f * x[p] - m), 1.f / s, p / S, p % S, hat, gc);
    }
    loss[0] = B > 0 ? (float)(tot * weight / B) : 0.f;
    return 0;
}
#endif
