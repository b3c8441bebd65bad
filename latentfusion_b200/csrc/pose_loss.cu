// Fused pose-loss head (SURVEY.md §8f-1).
//
// Replaces, per refinement iteration, the reference's
//   interpret_logits (recon/models.py:455-484: tanh, sigmoid, mask gate)
//   Camera.denormalize_depth (modules/geometry.py:555-558)
//   Camera.uncrop x2 (geometry.py:261-285: 2-D grid_sample to the 640x480 frame, nearest for depth,
//                     bilinear for mask logits, padding_mode='border')
//   default_pose_loss (pose/estimation.py:70-118) + pose/utils.py:81-117 reductions
// i.e. ~100 elementwise/reduction launches over [N,1,480,640] intermediates plus two
// grid_sampler_2d_backward launches that serialise on border-pixel atomics (1.5 ms each on B200),
// by two passes over the full frame:
//   pass 1: per-hypothesis partial sums  ->  the four loss terms
//   pass 2: d(terms)/d(depth logits, mask logits, viewport, translation_z): per-pixel gradients, gathered into the
//           crop maps by a row and a column pass (the taps are separable), every sum in a fixed order

#include "common.cuh"

namespace lf {

constexpr int kSums = 6;   // A=sum dl1, B=sum dl1*pm*tm, C=sum pm*tm, D=sum pm, E=sum pm*tm*valid, F=sum bce

struct LossGeom {
    int n, p, width, height;
    float range, base_off;    // z = (tanh(dl)+1)/2 * gate * range + (tz + base_off)
    int ps, hs, tzs;          // strides in floats: between crop pixels of a logit map, between hypotheses, between tz entries
    int premask;              // coarse search (PoseEstimator._render_observation, estimation.py:187-197): the crop's metric
                              // depth is multiplied by the crop's own sigmoid(mask) before it is pasted into the frame
};

struct PixelSample {
    // nearest tap (depth) and bilinear taps (mask logits) of one full-frame pixel in the P x P crop
    int near_idx;
    int i00, i01, i10, i11;
    float w00, w01, w10, w11;
    float fx, fy;             // bilinear fractions
    float mx, my;             // d(ix)/d(unclipped ix): 1 inside, 0 where border-clamped
    int x0in, y0in;           // whether the +1 taps are in range (weight is 0 otherwise)
};

// ATen grid_sampler (align_corners=False, padding border): unnormalize, clip to [0, P-1]
__device__ __forceinline__ float clip_coord(float g, int P, float& mult) {
    float ix = ((g + 1.f) * (float)P - 1.f) / 2.f;
    const float mxv = (float)(P - 1);
    if (ix <= 0.f) { ix = 0.f; mult = 0.f; }
    else if (ix >= mxv) { ix = mxv; mult = 0.f; }
    else mult = 1.f;
    return ix;
}

// one axis of a full-frame pixel's sample in the crop: gx = (X - v0)/(v1 - v0)*2 - 1 (geometry.py:281-282)
struct AxisSample {
    int i0, i1, near;         // bilinear taps (i1 == i0 at the far border) and the nearest tap
    int in;                   // whether the +1 tap is in range
    float f, w0, w1;          // fraction, tap weights (w1 = 0 at the far border)
    float m;                  // d(ix)/d(unclipped ix): 1 inside, 0 where border-clamped
    float ix;                 // the sample coordinate in [0, P-1]
};

__device__ __forceinline__ AxisSample axis_sample(float X, float v0, float v1, int P) {
    AxisSample a;
    const float gx = (X - v0) / (v1 - v0) * 2.f - 1.f;
    float ix = clip_coord(gx, P, a.m);
    // degenerate optimised viewport (zero width / NaN): the reference only propagates NaNs; keep the indices in range
    if (!isfinite(ix)) { ix = 0.f; a.m = 0.f; }
    a.ix = ix;
    a.near = (int)nearbyintf(ix);
    const float f0 = floorf(ix);
    a.i0 = (int)f0;
    a.f = ix - f0;
    a.in = (a.i0 + 1 < P);
    a.i1 = a.in ? a.i0 + 1 : a.i0;
    a.w0 = 1.f - a.f;
    a.w1 = a.in ? a.f : 0.f;
    return a;
}

__device__ __forceinline__ PixelSample make_sample(float X, float Y, const float* vp, int P, int ps) {
    PixelSample s;
    const AxisSample ax = axis_sample(X, vp[0], vp[2], P), ay = axis_sample(Y, vp[1], vp[3], P);
    s.mx = ax.m; s.my = ay.m;
    s.near_idx = (ay.near * P + ax.near) * ps;
    s.fx = ax.f; s.fy = ay.f;
    s.x0in = ax.in; s.y0in = ay.in;
    s.i00 = (ay.i0 * P + ax.i0) * ps; s.i01 = (ay.i0 * P + ax.i1) * ps;
    s.i10 = (ay.i1 * P + ax.i0) * ps; s.i11 = (ay.i1 * P + ax.i1) * ps;
    s.w00 = ax.w0 * ay.w0; s.w01 = ax.w1 * ay.w0; s.w10 = ax.w0 * ay.w1; s.w11 = ax.w1 * ay.w1;
    return s;
}

__device__ __forceinline__ float sigmoid_(float x) { return 1.f / (1.f + expf(-x)); }

struct PixelTerms { float z, pm, pd, dl1, td, tm, valid, ml, gate, th; };

__device__ __forceinline__ PixelTerms eval_pixel(const PixelSample& s, const float* __restrict__ dl,
                                                 const float* __restrict__ ml, float tdepth, float tmask,
                                                 float range, float base, int premask = 0) {
    PixelTerms t;
    t.th = tanhf(dl[s.near_idx]);
    t.gate = sigmoid_(ml[s.near_idx]) > 0.5f ? 1.f : 0.f;          // apply_mask (models.py:478-481)
    t.z = (t.th + 1.f) * 0.5f * t.gate * range + base;
    if (premask) t.z *= sigmoid_(ml[s.near_idx]);
    t.ml = s.w00 * ml[s.i00] + s.w01 * ml[s.i01] + s.w10 * ml[s.i10] + s.w11 * ml[s.i11];
    t.pm = sigmoid_(t.ml);
    t.pd = t.z * t.pm;
    t.valid = ((tdepth == 0.f) && (tmask > 0.1f)) ? 0.f : 1.f;
    t.tm = tmask;
    t.td = tdepth * tmask;                                          // Observation.prepare()
    t.dl1 = fabsf(t.pd - t.td) * t.valid;
    return t;
}

__global__ void __launch_bounds__(256)
pose_loss_sums_kernel(const LossGeom g, const float* __restrict__ dlog, const float* __restrict__ mlog,
                      const float* __restrict__ vp, const float* __restrict__ tz,
                      const float* __restrict__ tdepth, const float* __restrict__ tmask, float* __restrict__ part) {
    const int n = blockIdx.y;
    const int HW = g.width * g.height;
    const float* dl = dlog + (size_t)n * g.hs;
    const float* ml = mlog + (size_t)n * g.hs;
    const float base = tz[n * g.tzs] + g.base_off;
    float acc[kSums] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int px = blockIdx.x * blockDim.x + threadIdx.x; px < HW; px += gridDim.x * blockDim.x) {
        const int Y = px / g.width, X = px - Y * g.width;
        const PixelSample s = make_sample((float)X, (float)Y, vp + 4 * n, g.p, g.ps);
        const PixelTerms t = eval_pixel(s, dl, ml, tdepth[px], tmask[px], g.range, base, g.premask);
        acc[0] += t.dl1;
        acc[1] += t.dl1 * t.pm * t.tm;
        acc[2] += t.pm * t.tm;
        acc[3] += t.pm;
        acc[4] += t.pm * t.tm * t.valid;
        acc[5] += fmaxf(t.ml, 0.f) - t.ml * t.tm + log1pf(expf(-fabsf(t.ml)));   // BCE-with-logits
    }
    __shared__ float red[8][kSums];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < kSums; ++k) {
        const float r = warp_sum(acc[k]);
        if (lane == 0) red[warp][k] = r;
    }
    __syncthreads();
    if (threadIdx.x < kSums) {
        float r = 0.f;
        for (int w = 0; w < 8; ++w) r += red[w][threadIdx.x];
        part[((size_t)n * gridDim.x + blockIdx.x) * kSums + threadIdx.x] = r;
    }
}

// Adds the per-block partials of the two kernels around it in block order (no atomics: the same inputs give the same
// bits on every run) into sums[n][0..6], sums[n][6] = sum target_mask*valid, then
// terms[n] = (ov_depth, depth, iou, mask).
__global__ void pose_loss_terms_kernel(const LossGeom g, const float* __restrict__ part, int bx,
                                       const float* __restrict__ tpart, int tb, float* __restrict__ sums,
                                       float* __restrict__ terms) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= g.n) return;
    float* s = sums + n * 8;
    for (int k = 0; k < kSums; ++k) {
        float r = 0.f;
        for (int b = 0; b < bx; ++b) r += part[((size_t)n * bx + b) * kSums + k];
        s[k] = r;
    }
    float G = 0.f;
    for (int b = 0; b < tb; ++b) G += tpart[b];
    s[6] = G;
    const float HW = (float)(g.width * g.height);
    const float U = s[3] + G - s[4];
    terms[n * 4 + 0] = fmaxf(s[1], 1e-5f) / fmaxf(s[2], 1e-4f);            // pose/utils.py:111-117
    terms[n * 4 + 1] = s[0] / HW;
    terms[n * 4 + 2] = logf(fmaxf(U, 1e-4f)) - logf(fmaxf(s[4], 1e-4f));  // pose/utils.py:99-108
    terms[n * 4 + 3] = s[5] / HW;
}

__global__ void __launch_bounds__(256)
target_sum_kernel(const LossGeom g, const float* __restrict__ tdepth, const float* __restrict__ tmask, float* __restrict__ tpart) {
    const int HW = g.width * g.height;
    float a = 0.f;
    for (int px = blockIdx.x * blockDim.x + threadIdx.x; px < HW; px += gridDim.x * blockDim.x) {
        const float tm = tmask[px];
        a += ((tdepth[px] == 0.f) && (tm > 0.1f)) ? 0.f : tm;
    }
    a = warp_sum(a);
    __shared__ float red[8];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        float r = 0.f;
        for (int w = 0; w < 8; ++w) r += red[w];
        tpart[blockIdx.x] = r;
    }
}

__global__ void __launch_bounds__(256, 4)
pose_loss_bwd_kernel(const LossGeom g, const float* __restrict__ dlog, const float* __restrict__ mlog,
                     const float* __restrict__ vp, const float* __restrict__ tz,
                     const float* __restrict__ tdepth, const float* __restrict__ tmask,
                     const float* __restrict__ sums, const float* __restrict__ gterms,
                     float2* __restrict__ g_pix, float* __restrict__ vpart) {
    // pass 1 of the backward: every full-frame pixel's d(total)/d(sampled mask logit, depth logit) -> g_pix[n][px], and
    // this block's share of d/d(viewport, tz) -> vpart; pose_loss_rows/cols_kernel gather g_pix into the crop maps
    const int n = blockIdx.y;
    const int HW = g.width * g.height;
    const float* dl = dlog + (size_t)n * g.hs;
    const float* ml = mlog + (size_t)n * g.hs;
    const float base = tz[n * g.tzs] + g.base_off;
    const float* s = sums + n * 8;
    const float fHW = (float)HW;
    // d(total)/d(sums) from d(total)/d(terms)
    const float g_ov = gterms[n * 4 + 0], g_dep = gterms[n * 4 + 1], g_iou = gterms[n * 4 + 2], g_msk = gterms[n * 4 + 3];
    const float Cc = fmaxf(s[2], 1e-4f), Bc = fmaxf(s[1], 1e-5f);
    const float U = s[3] + s[6] - s[4];
    const float dA = g_dep / fHW;
    const float dB = (s[1] > 1e-5f) ? g_ov / Cc : 0.f;
    const float dC = (s[2] > 1e-4f) ? -g_ov * Bc / (Cc * Cc) : 0.f;
    const float dU = (U > 1e-4f) ? g_iou / U : 0.f;
    const float dD = dU;
    const float dE = ((s[4] > 1e-4f) ? -g_iou / s[4] : 0.f) - dU;
    const float dF = g_msk / fHW;
    const float vx0 = vp[4 * n], vy0 = vp[4 * n + 1], vw = vp[4 * n + 2] - vx0, vh = vp[4 * n + 3] - vy0;
    const float inv_vw = 1.f / vw, inv_vh = 1.f / vh, two_inv_vw = 2.f * inv_vw, two_inv_vh = 2.f * inv_vh;
    const float half_p = (float)g.p * 0.5f;            // d ix / d gx

    float a_tz = 0.f, a_vp[4] = {0.f, 0.f, 0.f, 0.f};
    for (int px = blockIdx.x * blockDim.x + threadIdx.x; px < HW; px += gridDim.x * blockDim.x) {
        const int Y = px / g.width, X = px - Y * g.width;
        const PixelSample smp = make_sample((float)X, (float)Y, vp + 4 * n, g.p, g.ps);
        const PixelTerms t = eval_pixel(smp, dl, ml, tdepth[px], tmask[px], g.range, base);
        float d_dl1 = dA + dB * t.pm * t.tm;
        float d_pm = dB * t.dl1 * t.tm + dC * t.tm + dD + dE * t.tm * t.valid;
        const float diff = t.pd - t.td;
        const float sgn = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
        const float d_pd = d_dl1 * t.valid * sgn;
        const float d_z = d_pd * t.pm;
        d_pm += d_pd * t.z;
        const float d_ml = d_pm * t.pm * (1.f - t.pm) + dF * (t.pm - t.tm);
        const float d_dlog = d_z * (1.f - t.th * t.th) * 0.5f * t.gate * g.range;
        a_tz += d_z;
        g_pix[(size_t)n * HW + px] = make_float2(d_ml, d_dlog);
        // d(ml_full)/d(ix, iy) -> viewport (ATen grid_sampler_2d_backward: gix uses the in-range taps only)
        const float m00 = ml[smp.i00], m01 = smp.x0in ? ml[smp.i01] : 0.f;
        const float m10 = smp.y0in ? ml[smp.i10] : 0.f, m11 = (smp.x0in && smp.y0in) ? ml[smp.i11] : 0.f;
        const float wy0 = 1.f - smp.fy, wy1 = smp.y0in ? smp.fy : 0.f;
        const float wx0 = 1.f - smp.fx, wx1 = smp.x0in ? smp.fx : 0.f;
        const float dml_dix = (smp.x0in ? (m01 - m00) : -m00) * wy0 + ((smp.x0in ? m11 : 0.f) - m10) * wy1;
        const float dml_diy = (smp.y0in ? (m10 - m00) : -m00) * wx0 + ((smp.y0in ? m11 : 0.f) - m01) * wx1;
        const float gix = d_ml * dml_dix * smp.mx * half_p;
        const float giy = d_ml * dml_diy * smp.my * half_p;
        // gx = (X - vx0)/vw*2 - 1:  d gx / d vx0 = 2*(rx - 1)/vw,  d gx / d vx1 = -2*rx/vw  with rx = (X - vx0)/vw
        const float rx = ((float)X - vx0) * inv_vw, ry = ((float)Y - vy0) * inv_vh;
        const float tx = gix * two_inv_vw, ty = giy * two_inv_vh;
        a_vp[0] += tx * (rx - 1.f);
        a_vp[2] -= tx * rx;
        a_vp[1] += ty * (ry - 1.f);
        a_vp[3] -= ty * ry;
    }
    __shared__ float red[8][5];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float v5[5] = {a_vp[0], a_vp[1], a_vp[2], a_vp[3], a_tz};
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const float r = warp_sum(v5[k]);
        if (lane == 0) red[warp][k] = r;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        float r = 0.f;
        for (int w = 0; w < 8; ++w) r += red[w][threadIdx.x];
        vpart[((size_t)n * gridDim.x + blockIdx.x) * 5 + threadIdx.x] = r;
    }
}

// The pixels whose sample along one axis has its first bilinear tap in [t0, t1]: a contiguous range [lo, hi), as the
// tap is non-decreasing in the pixel coordinate for a viewport of positive extent (clamping and float rounding are
// monotone).  Any other viewport (flipped, empty, NaN) scans the whole axis.
__device__ __forceinline__ void tap_range(int t0, int t1, float v0, float v1, int P, int len, int& lo, int& hi) {
    if (!((v1 - v0) > 0.f)) { lo = 0; hi = len; return; }
    auto first = [&](int t) {               // first pixel whose tap is >= t
        int a = 0, b = len;
        while (a < b) {
            const int mid = (a + b) >> 1;
            if (axis_sample((float)mid, v0, v1, P).i0 >= t) b = mid; else a = mid + 1;
        }
        return a;
    };
    lo = first(t0);
    hi = first(t1 + 1);
}

// The pixels at the two ends of an axis whose sample is clamped to the crop border (coordinate 0, resp. P-1) give their
// whole value to the border texel, for the bilinear and the nearest tap alike.  A warp adds them up cooperatively
// (lane-strided partials, then a fixed shuffle tree), and the per-texel loops cover only the pixels in between:
// [lo_in, hi_in).  A viewport of non-positive extent keeps the full per-texel scans.
struct BorderSums { int lo_in, hi_in; float2 left, right; };

__device__ __forceinline__ BorderSums border_sums(const float2* src, int64_t stride, int len, float v0, float v1, int P) {
    BorderSums b;
    b.lo_in = 0; b.hi_in = len;
    b.left = b.right = make_float2(0.f, 0.f);
    if (!((v1 - v0) > 0.f)) return b;
    auto first = [&](float t, bool strict) {        // first pixel whose coordinate is > t (strict) or >= t
        int a = 0, e = len;
        while (a < e) {
            const int mid = (a + e) >> 1;
            const float ix = axis_sample((float)mid, v0, v1, P).ix;
            if (strict ? ix > t : ix >= t) e = mid; else a = mid + 1;
        }
        return a;
    };
    b.lo_in = first(0.f, true);
    b.hi_in = first((float)(P - 1), false);
    const int lane = threadIdx.x & 31;
    float lx = 0.f, ly = 0.f, rx = 0.f, ry = 0.f;
    for (int i = lane; i < b.lo_in; i += 32) { const float2 v = src[i * stride]; lx += v.x; ly += v.y; }
    for (int i = b.hi_in + lane; i < len; i += 32) { const float2 v = src[i * stride]; rx += v.x; ry += v.y; }
    b.left = make_float2(warp_sum(lx), warp_sum(ly));
    b.right = make_float2(warp_sum(rx), warp_sum(ry));
    return b;
}

// Sum over the in-between pixels of one texel: mask-logit values weighted by the texel's bilinear tap weight, and the
// depth-logit values of the pixels whose nearest tap is the texel, in increasing pixel order.
__device__ __forceinline__ float2 texel_sum(const float2* src, int64_t stride, int len, float v0, float v1, int P, int t,
                                            const BorderSums& b) {
    int lo, hi;
    tap_range(t - 1, t, v0, v1, P, len, lo, hi);
    lo = max(lo, b.lo_in);
    hi = min(hi, b.hi_in);
    float sml = 0.f, sdl = 0.f;
    for (int i = lo; i < hi; ++i) {
        const AxisSample a = axis_sample((float)i, v0, v1, P);
        const float w = (a.i0 == t ? a.w0 : 0.f) + (a.i1 == t ? a.w1 : 0.f);
        const float2 v = src[i * stride];
        sml += v.x * w;
        if (a.near == t) sdl += v.y;
    }
    if (t == 0) { sml += b.left.x; sdl += b.left.y; }
    if (t == P - 1) { sml += b.right.x; sdl += b.right.y; }
    return make_float2(sml, sdl);
}

// pass 2, one warp per (n, Y): rows[n][Y][tx] = x-gather of row Y of the per-pixel gradients into the crop columns.
__global__ void __launch_bounds__(256)
pose_loss_rows_kernel(const LossGeom g, const float* __restrict__ vp, const float2* __restrict__ g_pix,
                      float2* __restrict__ rows) {
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= (int64_t)g.n * g.height) return;              // (whole warps)
    const int n = (int)(row / g.height);
    const float v0 = vp[4 * n], v1 = vp[4 * n + 2];
    const float2* src = g_pix + row * g.width;
    const BorderSums b = border_sums(src, 1, g.width, v0, v1, g.p);
    for (int tx = threadIdx.x & 31; tx < g.p; tx += 32)
        rows[row * g.p + tx] = texel_sum(src, 1, g.width, v0, v1, g.p, tx, b);
}

// pass 3, one warp per (n, tx): the y-gather of column tx of `rows` into the crop maps, written to every texel in the
// inputs' layout; block 0 of each hypothesis adds the viewport / tz partials in block order.
__global__ void __launch_bounds__(256)
pose_loss_cols_kernel(const LossGeom g, const float* __restrict__ vp, const float2* __restrict__ rows,
                      const float* __restrict__ vpart, int bx, float* __restrict__ g_dl, float* __restrict__ g_ml,
                      float* __restrict__ g_vp, float* __restrict__ g_tz) {
    const int n = blockIdx.y;
    if (blockIdx.x == 0 && threadIdx.x < 5) {
        float r = 0.f;
        for (int b = 0; b < bx; ++b) r += vpart[((size_t)n * bx + b) * 5 + threadIdx.x];
        if (threadIdx.x < 4) g_vp[4 * n + threadIdx.x] = r;
        else g_tz[n * g.tzs] = r;
    }
    const int tx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (tx >= g.p) return;                                    // (whole warps)
    const float v0 = vp[4 * n + 1], v1 = vp[4 * n + 3];
    const float2* src = rows + (size_t)n * g.height * g.p + tx;
    const BorderSums b = border_sums(src, g.p, g.height, v0, v1, g.p);
    for (int ty = threadIdx.x & 31; ty < g.p; ty += 32) {
        const float2 v = texel_sum(src, g.p, g.height, v0, v1, g.p, ty, b);
        const size_t e = (size_t)n * g.hs + (size_t)(ty * g.p + tx) * g.ps;
        g_ml[e] = v.x;
        g_dl[e] = v.y;
    }
}

// blocks along x for a (bx, n) grid of grid-stride CTAs: as many as are co-resident (occupancy x SMs), so that the
// launch is ONE balanced wave (600 CTAs on 444 slots ran as two waves, the second one nearly empty)
template <typename K>
static int blocks_x(K kernel, int n, int HW) {
    static int per_sm = 0;                      // per kernel instantiation (K is a distinct function type per kernel)
    if (per_sm == 0) {
        int v = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, kernel, 256, 0) != cudaSuccess || v < 1) v = 2;
        per_sm = v;
    }
    int bx = per_sm * sm_count() / max(1, n);
    bx = max(1, min(bx, (HW + 255) / 256));
    return bx;
}

static int loss_geom(const lf_loss_desc* d, LossGeom& g) {
    LF_CHECK_ARG(d != nullptr, "pose_loss: null descriptor");
    LF_CHECK_ARG(d->n > 0 && d->p > 1 && d->width > 0 && d->height > 0, "pose_loss: bad extents");
    g.n = d->n; g.p = d->p; g.width = d->width; g.height = d->height;
    g.range = 2.f * d->z_span + 2.f * d->eps;          // (zfar + eps) - (znear - eps)
    g.base_off = -d->z_span - d->eps;                  // znear - eps = tz - z_span - eps
    g.premask = 0;
    LF_CHECK_ARG(d->pix_stride >= 0 && d->hyp_stride >= 0 && d->tz_stride >= 0, "pose_loss: negative stride");
    g.ps = d->pix_stride > 0 ? d->pix_stride : 1;
    g.hs = d->hyp_stride > 0 ? d->hyp_stride : d->p * d->p * g.ps;
    g.tzs = d->tz_stride > 0 ? d->tz_stride : 1;
    LF_CHECK_ARG((int64_t)g.hs >= (int64_t)(d->p * d->p - 1) * g.ps + 1, "pose_loss: hypothesis stride smaller than one logit map");
    return LF_OK;
}

// Workspaces (no atomics anywhere, so that the same inputs give the same bits on every run):
//   forward : per-block partial sums of the loss kernel [n][bx][6] and of the target kernel [tb]
//   backward: per-pixel gradients [n][H][W] float2, row sums [n][H][P] float2, per-block viewport/tz partials [n][bx][5]
static int target_blocks(int HW) { return min(2 * sm_count(), (HW + 255) / 256); }

static int64_t fwd_ws_floats(const LossGeom& g) {
    const int HW = g.width * g.height;
    return (int64_t)g.n * blocks_x(pose_loss_sums_kernel, g.n, HW) * kSums + target_blocks(HW);
}

static int64_t bwd_ws_floats(const LossGeom& g) {
    const int HW = g.width * g.height;
    return 2 * (int64_t)g.n * HW + 2 * (int64_t)g.n * g.height * g.p + (int64_t)g.n * blocks_x(pose_loss_bwd_kernel, g.n, HW) * 5;
}

static int loss_fwd(const LossGeom& g, const float* depth_logits, const float* mask_logits, const float* viewport,
                    const float* tz, const float* target_depth, const float* target_mask, float* sums, float* terms,
                    void* workspace, cudaStream_t st) {
    const int HW = g.width * g.height;
    const int bx = blocks_x(pose_loss_sums_kernel, g.n, HW), tb = target_blocks(HW);
    float* part = (float*)workspace;
    float* tpart = part + (size_t)g.n * bx * kSums;
    target_sum_kernel<<<tb, 256, 0, st>>>(g, target_depth, target_mask, tpart);
    pose_loss_sums_kernel<<<dim3(bx, g.n), 256, 0, st>>>(g, depth_logits, mask_logits, viewport, tz, target_depth, target_mask, part);
    pose_loss_terms_kernel<<<(g.n + 63) / 64, 64, 0, st>>>(g, part, bx, tpart, tb, sums, terms);
    LF_RETURN_LAUNCH();
}

}  // namespace lf

using namespace lf;

extern "C" int64_t lf_pose_loss_fwd_ws(const lf_loss_desc* desc) {
    LossGeom g;
    if (int e = loss_geom(desc, g)) return e;
    return 4 * fwd_ws_floats(g);
}

extern "C" int64_t lf_pose_loss_bwd_ws(const lf_loss_desc* desc) {
    LossGeom g;
    if (int e = loss_geom(desc, g)) return e;
    return 4 * bwd_ws_floats(g);
}

extern "C" int lf_pose_loss_fwd(const lf_loss_desc* desc, const float* depth_logits, const float* mask_logits,
                                const float* viewport, const float* tz, const float* target_depth,
                                const float* target_mask, float* sums, float* terms, void* workspace, void* stream) {
    LossGeom g;
    if (int e = loss_geom(desc, g)) return e;
    LF_CHECK_ARG(depth_logits && mask_logits && viewport && tz && target_depth && target_mask && sums && terms && workspace,
                 "pose_loss_fwd: null pointer");
    return loss_fwd(g, depth_logits, mask_logits, viewport, tz, target_depth, target_mask, sums, terms, workspace,
                    (cudaStream_t)stream);
}

// Forward-only scoring for the coarse pose search (CrossEntropyPoseEstimator, reference estimation.py:187-197 +
// :70-118): same four terms, with the search's extra crop-space mask factor on the rendered depth.
extern "C" int lf_pose_loss_search_fwd(const lf_loss_desc* desc, const float* depth_logits, const float* mask_logits,
                                       const float* viewport, const float* tz, const float* target_depth,
                                       const float* target_mask, float* sums, float* terms, void* workspace,
                                       void* stream) {
    LossGeom g;
    if (int e = loss_geom(desc, g)) return e;
    g.premask = 1;
    LF_CHECK_ARG(depth_logits && mask_logits && viewport && tz && target_depth && target_mask && sums && terms && workspace,
                 "pose_loss_search_fwd: null pointer");
    return loss_fwd(g, depth_logits, mask_logits, viewport, tz, target_depth, target_mask, sums, terms, workspace,
                    (cudaStream_t)stream);
}

extern "C" int lf_pose_loss_bwd(const lf_loss_desc* desc, const float* depth_logits, const float* mask_logits,
                                const float* viewport, const float* tz, const float* target_depth,
                                const float* target_mask, const float* sums, const float* grad_terms,
                                float* grad_depth_logits, float* grad_mask_logits, float* grad_viewport,
                                float* grad_tz, void* workspace, void* stream) {
    LossGeom g;
    if (int e = loss_geom(desc, g)) return e;
    LF_CHECK_ARG(depth_logits && mask_logits && viewport && tz && target_depth && target_mask && sums && grad_terms &&
                 grad_depth_logits && grad_mask_logits && grad_viewport && grad_tz && workspace,
                 "pose_loss_bwd: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const int HW = g.width * g.height;
    const int bx = blocks_x(pose_loss_bwd_kernel, g.n, HW);
    float2* g_pix = (float2*)workspace;
    float2* rows = g_pix + (size_t)g.n * HW;
    float* vpart = (float*)(rows + (size_t)g.n * g.height * g.p);
    pose_loss_bwd_kernel<<<dim3(bx, g.n), 256, 0, st>>>(g, depth_logits, mask_logits, viewport, tz, target_depth,
                                                      target_mask, sums, grad_terms, g_pix, vpart);
    pose_loss_rows_kernel<<<(unsigned)(((int64_t)g.n * g.height * 32 + 255) / 256), 256, 0, st>>>(g, viewport, g_pix, rows);
    pose_loss_cols_kernel<<<dim3((g.p * 32 + 255) / 256, g.n), 256, 0, st>>>(g, viewport, rows, vpart, bx,
                                                                            grad_depth_logits, grad_mask_logits,
                                                                            grad_viewport, grad_tz);
    LF_RETURN_LAUNCH();
}
