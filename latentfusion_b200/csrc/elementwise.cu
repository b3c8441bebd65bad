// Memory-bound helpers of the path: Interpolate (x2 / x0.5, nearest or linear), view-axis pooling
// fusers, ConvGRU gate math.  All channels-last fp32; one thread per (position, 4 channels) where C%4==0.
#include "common.cuh"

namespace lf {

// ---------------------------------------------------------------------------------------------
// Interpolate (modules/__init__.py:18-33 -> F.interpolate(scale_factor, mode, align_corners=False)).
//   nearest: src = floor(dst / scale)         linear: src = (dst + .5)/scale - .5, clamped at 0
// Each output element is a tensor-product of <= 2 taps per axis; the backward gathers through the same taps.
// ---------------------------------------------------------------------------------------------
struct Tap { int i0, i1; float w0, w1; };

__device__ __forceinline__ Tap axis_tap(int o, int in_size, int mode, int factor) {
    Tap t;
    if (factor == 1) { t.i0 = t.i1 = o; t.w0 = 1.f; t.w1 = 0.f; return t; }
    if (mode == 0) {
        t.i0 = factor > 0 ? o / 2 : min(o * 2, in_size - 1);
        t.i1 = t.i0; t.w0 = 1.f; t.w1 = 0.f;
        return t;
    }
    const float inv_scale = factor > 0 ? 0.5f : 2.f;
    float src = ((float)o + 0.5f) * inv_scale - 0.5f;
    if (src < 0.f) src = 0.f;
    t.i0 = (int)src;
    t.i1 = t.i0 + (t.i0 < in_size - 1 ? 1 : 0);
    t.w1 = src - (float)t.i0;
    t.w0 = 1.f - t.w1;
    return t;
}

struct InterpGeom {
    int n, d, h, w, c;          // input extent
    int od, oh, ow;             // output extent
    int fd, fh, fw;             // per-axis factor: 1 (untouched), 2, -2
    int mode;
};

template <int VEC>
__global__ void interp_kernel(const InterpGeom g, const float* __restrict__ x, float* __restrict__ y) {
    // VEC = 4 when C % 4 == 0: one thread moves 4 channels with 128-bit loads/stores.
    const int cv = g.c / VEC;
    const int64_t total = (int64_t)g.n * g.od * g.oh * g.ow * cv;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = e;
        const int c = (int)(r % cv) * VEC; r /= cv;
        const int ox = (int)(r % g.ow); r /= g.ow;
        const int oy = (int)(r % g.oh); r /= g.oh;
        const int oz = (int)(r % g.od); r /= g.od;
        const int n = (int)r;
        const Tap tz = axis_tap(oz, g.d, g.mode, g.fd);
        const Tap ty = axis_tap(oy, g.h, g.mode, g.fh);
        const Tap tx = axis_tap(ox, g.w, g.mode, g.fw);
        const int64_t base = (int64_t)n * g.d;
        float acc[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
#pragma unroll
        for (int a = 0; a < 2; ++a) {
            const float wz = a ? tz.w1 : tz.w0; const int iz = a ? tz.i1 : tz.i0;
            if (wz == 0.f) continue;
#pragma unroll
            for (int b = 0; b < 2; ++b) {
                const float wy = b ? ty.w1 : ty.w0; const int iy = b ? ty.i1 : ty.i0;
                if (wy == 0.f) continue;
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const float wx = q ? tx.w1 : tx.w0; const int ix = q ? tx.i1 : tx.i0;
                    if (wx == 0.f) continue;
                    const float wgt = wz * wy * wx;
                    const int64_t idx = (((base + iz) * g.h + iy) * g.w + ix) * g.c + c;
                    if (VEC == 4) {
                        const float4 t = ldg4(x + idx);
                        acc[0] += wgt * t.x; acc[1] += wgt * t.y; acc[2] += wgt * t.z; acc[3] += wgt * t.w;
                    } else {
                        acc[0] += wgt * x[idx];
                    }
                }
            }
        }
        if (VEC == 4) *reinterpret_cast<float4*>(y + e * 4) = make_float4(acc[0], acc[1], acc[2], acc[3]);
        else y[e] = acc[0];
    }
}

// The weight output o gives input index i along one axis through its forward taps (both taps count when a border
// clamp makes them coincide).  Only outputs in gather_lo(i) .. gather_hi(i) can reach i: 2i-1 .. 2i+2 when upsampling
// (the linear stencil; nearest uses 2i, 2i+1), i/2 when downsampling (taps 2o, 2o+1 linear, 2o nearest).
__device__ __forceinline__ float tap_weight(int o, int i, int in_size, int mode, int factor) {
    const Tap t = axis_tap(o, in_size, mode, factor);
    return (t.i0 == i ? t.w0 : 0.f) + (t.i1 == i ? t.w1 : 0.f);
}
__device__ __forceinline__ int gather_lo(int i, int factor) { return max(factor == 1 ? i : (factor > 0 ? 2 * i - 1 : i / 2), 0); }
__device__ __forceinline__ int gather_hi(int i, int out_size, int factor) {
    return min(factor == 1 ? i : (factor > 0 ? 2 * i + 2 : i / 2), out_size - 1);
}

// Backward as a gather: each element of gx sums its gradient contributions in a fixed order, so the result does not
// depend on scheduling (a scatter with float atomics would add them in a different order on every run).
template <int VEC>
__global__ void interp_bwd_kernel(const InterpGeom g, const float* __restrict__ gy, float* __restrict__ gx) {
    const int cv = g.c / VEC;
    const int64_t total = (int64_t)g.n * g.d * g.h * g.w * cv;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = e;
        const int c = (int)(r % cv) * VEC; r /= cv;
        const int ix = (int)(r % g.w); r /= g.w;
        const int iy = (int)(r % g.h); r /= g.h;
        const int iz = (int)(r % g.d); r /= g.d;
        const int n = (int)r;
        const int64_t base = (int64_t)n * g.od;
        float acc[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
        for (int oz = gather_lo(iz, g.fd); oz <= gather_hi(iz, g.od, g.fd); ++oz) {
            const float wz = tap_weight(oz, iz, g.d, g.mode, g.fd);
            if (wz == 0.f) continue;
            for (int oy = gather_lo(iy, g.fh); oy <= gather_hi(iy, g.oh, g.fh); ++oy) {
                const float wy = tap_weight(oy, iy, g.h, g.mode, g.fh);
                if (wy == 0.f) continue;
                for (int ox = gather_lo(ix, g.fw); ox <= gather_hi(ix, g.ow, g.fw); ++ox) {
                    const float wx = tap_weight(ox, ix, g.w, g.mode, g.fw);
                    if (wx == 0.f) continue;
                    const float wgt = wz * wy * wx;
                    const int64_t idx = (((base + oz) * g.oh + oy) * g.ow + ox) * g.c + c;
                    if (VEC == 4) {
                        const float4 t = ldg4(gy + idx);
                        acc[0] += wgt * t.x; acc[1] += wgt * t.y; acc[2] += wgt * t.z; acc[3] += wgt * t.w;
                    } else {
                        acc[0] += wgt * gy[idx];
                    }
                }
            }
        }
        if (VEC == 4) *reinterpret_cast<float4*>(gx + e * 4) = make_float4(acc[0], acc[1], acc[2], acc[3]);
        else gx[e] = acc[0];
    }
}

static int interp_geom(InterpGeom& g, int ndim, int n, int d, int h, int w, int c, int mode, int factor) {
    LF_CHECK_ARG(ndim == 2 || ndim == 3, "interp: ndim must be 2 or 3");
    LF_CHECK_ARG(factor == 2 || factor == -2, "interp: factor must be 2 or -2");
    LF_CHECK_ARG(mode == 0 || mode == 1, "interp: mode must be 0 (nearest) or 1 (linear)");
    LF_CHECK_ARG(n > 0 && d > 0 && h > 0 && w > 0 && c > 0, "interp: bad extents");
    g.n = n; g.d = d; g.h = h; g.w = w; g.c = c; g.mode = mode;
    g.fd = ndim == 3 ? factor : 1; g.fh = factor; g.fw = factor;
    auto osz = [&](int s, int f) { return f == 1 ? s : (f > 0 ? s * 2 : s / 2); };
    g.od = osz(d, g.fd); g.oh = osz(h, g.fh); g.ow = osz(w, g.fw);
    LF_CHECK_ARG(g.od > 0 && g.oh > 0 && g.ow > 0, "interp: output would be empty");
    return LF_OK;
}

// ---------------------------------------------------------------------------------------------
// view-axis pooling (recon/fusion.py:45-57): z[B][V][P][C] -> out[B][P][C]
// ---------------------------------------------------------------------------------------------
__global__ void fuse_pool_fwd_kernel(const float* __restrict__ z, float* __restrict__ out, int B, int V, int64_t PC, int kind) {
    const int64_t total = (int64_t)B * PC;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = e / PC, r = e - b * PC;
        const float* zp = z + b * V * PC + r;
        float res;
        if (kind == 0) {            // max
            res = zp[0];
            for (int v = 1; v < V; ++v) res = fmaxf(res, zp[(int64_t)v * PC]);
        } else if (kind == 1) {     // mean
            float s = 0.f;
            for (int v = 0; v < V; ++v) s += zp[(int64_t)v * PC];
            res = s / (float)V;
        } else if (kind == 2) {     // abs_max (functional.py:47-49): first index of the max |.|
            res = zp[0]; float best = fabsf(res);
            for (int v = 1; v < V; ++v) { const float t = zp[(int64_t)v * PC]; if (fabsf(t) > best) { best = fabsf(t); res = t; } }
        } else {                    // median: torch returns the LOWER median -> rank (V-1)/2
            const int want = (V - 1) / 2;
            res = zp[0];
            for (int v = 0; v < V; ++v) {
                const float t = zp[(int64_t)v * PC];
                int less = 0, eq = 0;
                for (int u = 0; u < V; ++u) { const float s2 = zp[(int64_t)u * PC]; less += s2 < t; eq += s2 == t; }
                if (less <= want && want < less + eq) { res = t; break; }
            }
        }
        out[e] = res;
    }
}

__global__ void fuse_pool_bwd_kernel(const float* __restrict__ gout, const float* __restrict__ z, float* __restrict__ gz,
                                     int B, int V, int64_t PC, int kind) {
    const int64_t total = (int64_t)B * PC;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = e / PC, r = e - b * PC;
        const float* zp = z + b * V * PC + r;
        float* gp = gz + b * V * PC + r;
        const float g = gout[e];
        if (kind == 1) {
            for (int v = 0; v < V; ++v) gp[(int64_t)v * PC] = g / (float)V;
            continue;
        }
        int sel = 0;
        if (kind == 0) {
            float best = zp[0];
            for (int v = 1; v < V; ++v) { const float t = zp[(int64_t)v * PC]; if (t > best) { best = t; sel = v; } }
        } else if (kind == 2) {
            float best = fabsf(zp[0]);
            for (int v = 1; v < V; ++v) { const float t = fabsf(zp[(int64_t)v * PC]); if (t > best) { best = t; sel = v; } }
        } else {
            const int want = (V - 1) / 2;
            for (int v = 0; v < V; ++v) {
                const float t = zp[(int64_t)v * PC];
                int less = 0, eq = 0;
                for (int u = 0; u < V; ++u) { const float s2 = zp[(int64_t)u * PC]; less += s2 < t; eq += s2 == t; }
                if (less <= want && want < less + eq) { sel = v; break; }
            }
        }
        for (int v = 0; v < V; ++v) gp[(int64_t)v * PC] = (v == sel) ? g : 0.f;
    }
}

// ---------------------------------------------------------------------------------------------
// ConvGRUCell gate math (modules/gru.py:36-43)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

__global__ void gru_gates1_kernel(const float* __restrict__ u_pre, const float* __restrict__ r_pre,
                                  const float* __restrict__ h, float* __restrict__ update, float* __restrict__ hr, int64_t n) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        update[e] = sigmoidf_(u_pre[e]);
        hr[e] = h[e] * sigmoidf_(r_pre[e]);
    }
}

__global__ void gru_gates2_kernel(const float* __restrict__ h, const float* __restrict__ update,
                                  const float* __restrict__ o, float* __restrict__ h_new, int64_t n) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const float u = update[e];
        h_new[e] = h[e] * (1.f - u) + o[e] * u;
    }
}

// backward of the two GRU gate kernels (modules/gru.py:38-41), one pass each
__global__ void gru_gates1_bwd_kernel(const float* __restrict__ g_update, const float* __restrict__ g_hr,
                                      const float* __restrict__ update, const float* __restrict__ r_pre,
                                      const float* __restrict__ h, float* __restrict__ g_u_pre, float* __restrict__ g_r_pre,
                                      float* __restrict__ g_h, int64_t n) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const float u = update[e], r = sigmoidf_(r_pre[e]), gh = g_hr[e];
        g_u_pre[e] = g_update[e] * u * (1.f - u);
        g_r_pre[e] = gh * h[e] * r * (1.f - r);
        g_h[e] = gh * r;
    }
}

__global__ void gru_gates2_bwd_kernel(const float* __restrict__ g, const float* __restrict__ h, const float* __restrict__ update,
                                      const float* __restrict__ o, float* __restrict__ g_h, float* __restrict__ g_update,
                                      float* __restrict__ g_o, int64_t n) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const float u = update[e], gg = g[e];
        g_h[e] = gg * (1.f - u);
        g_update[e] = gg * (o[e] - h[e]);
        g_o[e] = gg * u;
    }
}

// ConvLSTM gates (modules/lstm.py:41-56): gates [P][4H] channels-last = (i | f | o | g) pre-activations, c_cur [P][H]
//   c_next = sigmoid(f) * c_cur + sigmoid(i) * tanh(g);   h_next = sigmoid(o) * tanh(c_next)
__global__ void lstm_gates_fwd_kernel(const float* __restrict__ gates, const float* __restrict__ c_cur,
                                      float* __restrict__ h_next, float* __restrict__ c_next, int64_t P, int H) {
    const int64_t total = P * H;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t pos = e / H; const int c = (int)(e - pos * H);
        const float* gp = gates + pos * 4 * H + c;
        const float gi = sigmoidf_(gp[0]), gf = sigmoidf_(gp[H]), go = sigmoidf_(gp[2 * H]), gg = tanhf(gp[3 * H]);
        const float cn = gf * c_cur[e] + gi * gg;
        c_next[e] = cn;
        h_next[e] = go * tanhf(cn);
    }
}

__global__ void lstm_gates_bwd_kernel(const float* __restrict__ g_h, const float* __restrict__ g_c, const float* __restrict__ gates,
                                      const float* __restrict__ c_cur, float* __restrict__ g_gates, float* __restrict__ g_c_cur,
                                      int64_t P, int H) {
    const int64_t total = P * H;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t pos = e / H; const int c = (int)(e - pos * H);
        const float* gp = gates + pos * 4 * H + c;
        float* go_ = g_gates + pos * 4 * H + c;
        const float gi = sigmoidf_(gp[0]), gf = sigmoidf_(gp[H]), go = sigmoidf_(gp[2 * H]), gg = tanhf(gp[3 * H]);
        const float cc = c_cur[e], cn = gf * cc + gi * gg, tc = tanhf(cn);
        const float gh = g_h != nullptr ? g_h[e] : 0.f;
        const float dcn = (g_c != nullptr ? g_c[e] : 0.f) + gh * go * (1.f - tc * tc);
        go_[0] = dcn * gg * gi * (1.f - gi);
        go_[H] = dcn * cc * gf * (1.f - gf);
        go_[2 * H] = gh * tc * go * (1.f - go);
        go_[3 * H] = dcn * gi * (1.f - gg * gg);
        g_c_cur[e] = dcn * gf;
    }
}

// softmax over an outer axis followed by a weighted sum over it (channels-last):
//   BlendFuser (recon/fusion.py:92-96): scores [B][V][P], z [B][V][P][C]  -> w = softmax_V(scores), out[b][p][c] = sum_v w z
__global__ void softmax_blend_fwd_kernel(const float* __restrict__ scores, const float* __restrict__ z, float* __restrict__ wts,
                                         float* __restrict__ out, int B, int V, int64_t P, int C) {
    const int64_t total = (int64_t)B * P;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = e / P, pp = e - b * P;
        const float* sp = scores + b * V * P + pp;
        float m = -INFINITY;
        for (int v = 0; v < V; ++v) m = fmaxf(m, sp[(int64_t)v * P]);
        float den = 0.f;
        for (int v = 0; v < V; ++v) den += expf(sp[(int64_t)v * P] - m);
        for (int c = 0; c < C; ++c) out[e * C + c] = 0.f;
        for (int v = 0; v < V; ++v) {
            const float w = expf(sp[(int64_t)v * P] - m) / den;
            wts[(b * V + v) * P + pp] = w;
            const float* zp = z + ((b * V + v) * P + pp) * C;
            for (int c = 0; c < C; ++c) out[e * C + c] += w * zp[c];
        }
    }
}

__global__ void softmax_blend_bwd_kernel(const float* __restrict__ g_out, const float* __restrict__ g_wts,
                                         const float* __restrict__ wts, const float* __restrict__ z, float* __restrict__ g_scores,
                                         float* __restrict__ g_z, int B, int V, int64_t P, int C) {
    const int64_t total = (int64_t)B * P;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = e / P, pp = e - b * P;
        const float* go = g_out + e * C;
        float A = 0.f;
        for (int v = 0; v < V; ++v) {                 // up_v = <g_out, z_v> + g_wts_v;  A = sum_v w_v up_v
            const int64_t wi = (b * V + v) * P + pp;
            const float* zp = z + wi * C;
            float up = g_wts != nullptr ? g_wts[wi] : 0.f;
            for (int c = 0; c < C; ++c) up += go[c] * zp[c];
            g_scores[wi] = up;
            A += wts[wi] * up;
        }
        for (int v = 0; v < V; ++v) {
            const int64_t wi = (b * V + v) * P + pp;
            const float w = wts[wi];
            g_scores[wi] = w * (g_scores[wi] - A);
            if (g_z != nullptr) for (int c = 0; c < C; ++c) g_z[wi * C + c] = w * go[c];
        }
    }
}

// 'sum' projection (recon/models.py:436-437): x [N][D][Q][C] (Q = H*W) -> out [N][Q][C] = sum over depth
__global__ void depth_sum_fwd_kernel(const float* __restrict__ x, float* __restrict__ out, int N, int D, int64_t QC) {
    const int64_t total = (int64_t)N * QC;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t n = e / QC, r = e - n * QC;
        float s = 0.f;
        for (int d = 0; d < D; ++d) s += x[(n * D + d) * QC + r];
        out[e] = s;
    }
}

static unsigned ew_grid(int64_t total) {
    int64_t b = (total + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 32;
    return (unsigned)(b > cap ? cap : (b < 1 ? 1 : b));
}

}  // namespace lf

using namespace lf;

extern "C" int lf_interp_fwd(const float* x, float* y, int ndim, int n, int d, int h, int w, int c,
                             int mode, int factor, void* stream) {
    InterpGeom g;
    if (int e = interp_geom(g, ndim, n, d, h, w, c, mode, factor)) return e;
    LF_CHECK_ARG(x && y, "interp: null pointer");
    const int64_t total = (int64_t)g.n * g.od * g.oh * g.ow * g.c;
    if ((g.c & 3) == 0) interp_kernel<4><<<ew_grid(total / 4), 256, 0, (cudaStream_t)stream>>>(g, x, y);
    else interp_kernel<1><<<ew_grid(total), 256, 0, (cudaStream_t)stream>>>(g, x, y);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_interp_bwd(const float* gy, float* gx, int ndim, int n, int d, int h, int w, int c,
                             int mode, int factor, void* stream) {
    InterpGeom g;
    if (int e = interp_geom(g, ndim, n, d, h, w, c, mode, factor)) return e;
    LF_CHECK_ARG(gy && gx, "interp: null pointer");
    const int64_t total = (int64_t)g.n * g.d * g.h * g.w * g.c;
    if ((g.c & 3) == 0) interp_bwd_kernel<4><<<ew_grid(total / 4), 256, 0, (cudaStream_t)stream>>>(g, gy, gx);
    else interp_bwd_kernel<1><<<ew_grid(total), 256, 0, (cudaStream_t)stream>>>(g, gy, gx);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_fuse_pool_fwd(const float* z, float* out, int B, int V, int64_t P, int C, int kind, void* stream) {
    LF_CHECK_ARG(z && out, "fuse_pool: null pointer");
    LF_CHECK_ARG(B > 0 && V > 0 && P > 0 && C > 0 && kind >= 0 && kind <= 3, "fuse_pool: bad arguments");
    fuse_pool_fwd_kernel<<<ew_grid((int64_t)B * P * C), 256, 0, (cudaStream_t)stream>>>(z, out, B, V, P * C, kind);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_fuse_pool_bwd(const float* gout, const float* z, float* gz, int B, int V, int64_t P, int C,
                                int kind, void* stream) {
    LF_CHECK_ARG(gout && z && gz, "fuse_pool: null pointer");
    LF_CHECK_ARG(B > 0 && V > 0 && P > 0 && C > 0 && kind >= 0 && kind <= 3, "fuse_pool: bad arguments");
    fuse_pool_bwd_kernel<<<ew_grid((int64_t)B * P * C), 256, 0, (cudaStream_t)stream>>>(gout, z, gz, B, V, P * C, kind);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_gru_gates1(const float* u_pre, const float* r_pre, const float* h, float* update, float* hr,
                             int64_t numel, void* stream) {
    LF_CHECK_ARG(u_pre && r_pre && h && update && hr && numel > 0, "gru_gates1: bad arguments");
    gru_gates1_kernel<<<ew_grid(numel), 256, 0, (cudaStream_t)stream>>>(u_pre, r_pre, h, update, hr, numel);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_gru_gates1_bwd(const float* g_update, const float* g_hr, const float* update, const float* r_pre,
                                 const float* h, float* g_u_pre, float* g_r_pre, float* g_h, int64_t numel, void* stream) {
    LF_CHECK_ARG(g_update && g_hr && update && r_pre && h && g_u_pre && g_r_pre && g_h && numel > 0, "gru_gates1_bwd: bad arguments");
    gru_gates1_bwd_kernel<<<ew_grid(numel), 256, 0, (cudaStream_t)stream>>>(g_update, g_hr, update, r_pre, h, g_u_pre, g_r_pre, g_h, numel);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_gru_gates2_bwd(const float* g, const float* h, const float* update, const float* o, float* g_h,
                                 float* g_update, float* g_o, int64_t numel, void* stream) {
    LF_CHECK_ARG(g && h && update && o && g_h && g_update && g_o && numel > 0, "gru_gates2_bwd: bad arguments");
    gru_gates2_bwd_kernel<<<ew_grid(numel), 256, 0, (cudaStream_t)stream>>>(g, h, update, o, g_h, g_update, g_o, numel);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_lstm_gates_fwd(const float* gates, const float* c_cur, float* h_next, float* c_next, int64_t positions,
                                 int hidden, void* stream) {
    LF_CHECK_ARG(gates && c_cur && h_next && c_next && positions > 0 && hidden > 0, "lstm_gates: bad arguments");
    lstm_gates_fwd_kernel<<<ew_grid(positions * hidden), 256, 0, (cudaStream_t)stream>>>(gates, c_cur, h_next, c_next, positions, hidden);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_lstm_gates_bwd(const float* g_h, const float* g_c, const float* gates, const float* c_cur, float* g_gates,
                                 float* g_c_cur, int64_t positions, int hidden, void* stream) {
    LF_CHECK_ARG(gates && c_cur && g_gates && g_c_cur && positions > 0 && hidden > 0, "lstm_gates_bwd: bad arguments");
    lstm_gates_bwd_kernel<<<ew_grid(positions * hidden), 256, 0, (cudaStream_t)stream>>>(g_h, g_c, gates, c_cur, g_gates, g_c_cur,
                                                                                     positions, hidden);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_softmax_blend_fwd(const float* scores, const float* z, float* weights, float* out, int b, int v, int64_t p,
                                    int c, void* stream) {
    LF_CHECK_ARG(scores && z && weights && out && b > 0 && v > 0 && p > 0 && c > 0, "softmax_blend: bad arguments");
    softmax_blend_fwd_kernel<<<ew_grid((int64_t)b * p), 256, 0, (cudaStream_t)stream>>>(scores, z, weights, out, b, v, p, c);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_softmax_blend_bwd(const float* g_out, const float* g_weights, const float* weights, const float* z,
                                    float* g_scores, float* g_z, int b, int v, int64_t p, int c, void* stream) {
    LF_CHECK_ARG(g_out && weights && z && g_scores && b > 0 && v > 0 && p > 0 && c > 0, "softmax_blend_bwd: bad arguments");
    softmax_blend_bwd_kernel<<<ew_grid((int64_t)b * p), 256, 0, (cudaStream_t)stream>>>(g_out, g_weights, weights, z, g_scores, g_z,
                                                                                     b, v, p, c);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_depth_sum_fwd(const float* x, float* out, int n, int d, int64_t hw, int c, void* stream) {
    LF_CHECK_ARG(x && out && n > 0 && d > 0 && hw > 0 && c > 0, "depth_sum: bad arguments");
    depth_sum_fwd_kernel<<<ew_grid((int64_t)n * hw * c), 256, 0, (cudaStream_t)stream>>>(x, out, n, d, hw * c);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_gru_gates2(const float* h, const float* update, const float* o, float* h_new,
                             int64_t numel, void* stream) {
    LF_CHECK_ARG(h && update && o && h_new && numel > 0, "gru_gates2: bad arguments");
    gru_gates2_kernel<<<ew_grid(numel), 256, 0, (cudaStream_t)stream>>>(h, update, o, h_new, numel);
    LF_RETURN_LAUNCH();
}

// ------------------------------------------------------------------------------------------------
// Output heads of the render decoder (recon/models.py:331-338, :448-452): several 1x1 Equalized convs with 1-3
// output channels each, concatenated along channels.  As convolutions they are GEMMs with N = 1..3 — 52 us each on
// the implicit-GEMM kernels for 17 MB of input.  Here: one pass over x for ALL heads, exact fp32.
//   y[pos][h] = scale * sum_c x[pos][c] * w[h][c] + b[h]            h < H <= 8, C % 4 == 0, C <= 256
// LPV = C/4 lanes share a position (128-bit coalesced loads), partial dot products are xor-shuffled together.
// ------------------------------------------------------------------------------------------------
namespace lf {

constexpr int HEADS_MAX = 8;

__global__ void __launch_bounds__(256)
heads_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                 float* __restrict__ y, int64_t positions, int C, int H, int lg, float scale) {
    extern __shared__ float sw[];                  // [H][C]
    for (int i = threadIdx.x; i < H * C; i += blockDim.x) sw[i] = w[i];
    __syncthreads();
    const int q4 = C >> 2;
    const int64_t units = positions * q4, units_pad = (units + 31) & ~(int64_t)31;
    for (int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; u < units_pad; u += (int64_t)gridDim.x * blockDim.x) {
        const bool live = u < units;
        const int64_t uu = live ? u : units - 1;
        const int64_t pos = uu >> lg;
        const int q = (int)(uu & (q4 - 1));
        const float4 xv = ldg4(x + uu * 4);
        float acc[HEADS_MAX];
#pragma unroll
        for (int h = 0; h < HEADS_MAX; ++h) {
            if (h < H) {
                const float4 wv = *reinterpret_cast<const float4*>(sw + h * C + q * 4);
                float d = xv.x * wv.x + xv.y * wv.y + xv.z * wv.z + xv.w * wv.w;
                for (int s = 1; s < q4; s <<= 1) d += __shfl_xor_sync(0xffffffffu, d, s);
                acc[h] = d;
            }
        }
        if (live && q == 0) {
#pragma unroll
            for (int h = 0; h < HEADS_MAX; ++h)
                if (h < H) y[pos * H + h] = acc[h] * scale + (bias != nullptr ? bias[h] : 0.f);
        }
    }
}

// gx[pos][c] = scale * sum_h g[pos][h] * w[h][c]
__global__ void __launch_bounds__(256)
heads_bwd_kernel(const float* __restrict__ g, const float* __restrict__ w, float* __restrict__ gx,
                 int64_t positions, int C, int H, int lg, float scale) {
    extern __shared__ float sw[];
    for (int i = threadIdx.x; i < H * C; i += blockDim.x) sw[i] = w[i] * scale;
    __syncthreads();
    const int q4 = C >> 2;
    const int64_t units = positions * q4;
    for (int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; u < units; u += (int64_t)gridDim.x * blockDim.x) {
        const int64_t pos = u >> lg;
        const int q = (int)(u & (q4 - 1));
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int h = 0; h < H; ++h) {
            const float gv = __ldg(g + pos * H + h);
            const float4 wv = *reinterpret_cast<const float4*>(sw + h * C + q * 4);
            o.x += gv * wv.x; o.y += gv * wv.y; o.z += gv * wv.z; o.w += gv * wv.w;
        }
        *reinterpret_cast<float4*>(gx + u * 4) = o;
    }
}

static int heads_check(int64_t positions, int c, int h, int& lg) {
    LF_CHECK_ARG(positions > 0 && h >= 1 && h <= HEADS_MAX, "heads: need 1..%d output channels", HEADS_MAX);
    const int q4 = c >> 2;
    LF_CHECK_ARG(c >= 4 && (c & 3) == 0 && (q4 & (q4 - 1)) == 0 && q4 <= 32, "heads: Cin must be 4 * 2^k <= 128");
    lg = 0;
    while ((1 << lg) < q4) ++lg;
    return LF_OK;
}

}  // namespace lf

extern "C" int lf_heads_fwd(const float* x, const float* w, const float* bias, float* y, int64_t positions, int c, int h,
                            float scale, void* stream) {
    LF_CHECK_ARG(x && w && y, "heads_fwd: null pointer");
    int lg;
    if (int e = lf::heads_check(positions, c, h, lg)) return e;
    const int64_t units = positions * (c >> 2);
    int64_t blocks = (units + 255) / 256;
    const int64_t cap = (int64_t)lf::sm_count() * 16;
    if (blocks > cap) blocks = cap;
    lf::heads_fwd_kernel<<<(unsigned)blocks, 256, (size_t)h * c * sizeof(float), (cudaStream_t)stream>>>(
        x, w, bias, y, positions, c, h, lg, scale);
    LF_RETURN_LAUNCH();
}

extern "C" int lf_heads_bwd(const float* g, const float* w, float* gx, int64_t positions, int c, int h, float scale,
                            void* stream) {
    LF_CHECK_ARG(g && w && gx, "heads_bwd: null pointer");
    int lg;
    if (int e = lf::heads_check(positions, c, h, lg)) return e;
    const int64_t units = positions * (c >> 2);
    int64_t blocks = (units + 255) / 256;
    const int64_t cap = (int64_t)lf::sm_count() * 16;
    if (blocks > cap) blocks = cap;
    lf::heads_bwd_kernel<<<(unsigned)blocks, 256, (size_t)h * c * sizeof(float), (cudaStream_t)stream>>>(
        g, w, gx, positions, c, h, lg, scale);
    LF_RETURN_LAUNCH();
}
