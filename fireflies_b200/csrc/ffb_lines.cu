// Line and depth rasterisers for sm_100a (SURVEY.md section 8(f) row 2).
//
// Replaces (reference paths relative to the Fireflies tree):
//   fireflies/graphics/rasterization.py:107-153  rasterize_lines  (dense [L,H,W]; the epipolar-line regulariser of
//                                                Laser.render_epipolar_lines, projection/laser.py:298-325, and the
//                                                L1(softor, sum) loop of test_line_reg, rasterization.py:684-697)
//   fireflies/graphics/rasterization.py:66-104   rasterize_depth  (dense [N,H,W])
//   fireflies/graphics/rasterization.py:538-549  subsampled_point_raster (soft-OR over the points per pyramid level)
//   + the torch autograd of those w.r.t. `lines` / `points` / `depth_vals`.
//
// Design: HBM-bound elementwise / gather work, no tensor cores.  The dense kernels exist for API compatibility
// ([L,H,W] is what the reference returns).  The fused kernels produce what every caller reduces to next -- sum and
// soft-OR over the lines -- in one pass: a warp owns 8 rows x 32 columns of the texture, walks the line table staged
// in shared memory, skips lines whose segment is farther from its block than the radius where exp(-(d2^2)/sigma^2)
// underflows (warp-uniform), and writes every texel once with 128-byte row stores (8 B/texel instead of 12 L B/texel).
// The backward runs the same walk twice: pass 1 rebuilds the per-texel soft-OR product with torch.prod's zero
// bookkeeping (texels that lie exactly on a line have g = 1), pass 2 forms dL/dg per (texel, line), reduces the four
// end-point derivatives with warp shuffles and issues one shared-memory atomic per (warp, line), one global atomic
// per (CTA, line).
#include "ffb_common.cuh"

namespace ffb {
namespace lines {

constexpr int CTA = 256;       // 8 warps: 64 rows x 32 columns per CTA
constexpr int WROWS = 8;       // rows per warp
constexpr int TROWS = 64;
constexpr int TCOLS = 32;
constexpr int CHUNK = 128;     // lines staged per pass
static_assert(CTA == 32 * (TROWS / WROWS), "one warp per WROWS x TCOLS block of the CTA tile");
static_assert(CHUNK <= CTA, "stage_lines and the dl_s zeroing give each staged line one thread");

struct Seg {
    float ax, ay, bx, by;      // end points * texture_size
};

// squared distance of texel (x, y) to the segment, op for op as the reference (rasterization.py:140-151); t0 is returned
// for the backward's branch selection
__device__ __forceinline__ float seg_dist2(float x, float y, const Seg& s, float& t0, float& qx, float& qy) {
    const float pax = x - s.ax, pay = y - s.ay;
    const float pbx = x - s.bx, pby = y - s.by;
    const float mx = s.bx - s.ax, my = s.by - s.ay;
    const float dot = __fadd_rn(__fmul_rn(pax, mx), __fmul_rn(pay, my));
    const float mm = __fadd_rn(__fadd_rn(__fmul_rn(mx, mx), __fmul_rn(my, my)), 1.1920928955078125e-07f);   // torch.finfo().eps
    t0 = __fdiv_rn(dot, mm);
    if (t0 <= 0.f) { qx = pax; qy = pay; }
    else if (t0 >= 1.f) { qx = pbx; qy = pby; }
    else {
        qx = x - __fadd_rn(s.ax, __fmul_rn(t0, mx));
        qy = y - __fadd_rn(s.ay, __fmul_rn(t0, my));
    }
    return __fadd_rn(__fmul_rn(qx, qx), __fmul_rn(qy, qy));
}
__device__ __forceinline__ float line_g(float d2, float sig2) {
    const float w = __fdiv_rn(__fmul_rn(d2, d2), sig2);
    return w > 87.f ? 0.f : exp_neg(w);
}
// conservative: can any texel of the block [x0, x0+w) x [y0, y0+h) be closer to the segment than sqrt(cut2)?
__device__ __forceinline__ bool seg_near_block(const Seg& s, float x0, float y0, float w, float h, float cut) {
    const float cx = x0 + 0.5f * (w - 1.f), cy = y0 + 0.5f * (h - 1.f);
    float t0, qx, qy;
    const float d2 = seg_dist2(cx, cy, s, t0, qx, qy);
    const float r = 0.5f * sqrtf(w * w + h * h) + cut + 1.f;
    return !(d2 > r * r);       // NaN end points stay in (and produce the reference's NaNs)
}

__global__ void __launch_bounds__(256) dense_fwd_kernel(const float* __restrict__ lines, int L, int ts0, int ts1, float sig2,
                                                        float* __restrict__ out) {
    const size_t frame = (size_t)ts0 * ts1, total = frame * L;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int l = (int)(i / frame);
        const size_t t = i - (size_t)l * frame;
        const int r = (int)(t / ts0), c = (int)(t - (size_t)r * ts0);
        const float4 e = __ldg(reinterpret_cast<const float4*>(lines) + l);
        const Seg s = {e.x * (float)ts0, e.y * (float)ts1, e.z * (float)ts0, e.w * (float)ts1};
        float t0, qx, qy;
        out[i] = line_g(seg_dist2((float)c, (float)r, s, t0, qx, qy), sig2);
    }
}

// d out / d (segment end points, texture units) for one texel, weighted by `coef` and accumulated:
//   g = exp(-d2^2 / sig2)  =>  dg/dd2 = -2 d2 g / sig2;   d d2 / d a = -2 (1 - t) q,  d d2 / d b = -2 t q  with t = clamp(t0, 0, 1)
// (the term through t0 itself is 2 (q.m) dt0 = 2 t0 eps dt0, nine orders below the others, and is dropped)
__device__ __forceinline__ void seg_accum(float coef, float g, float d2, float t0, float qx, float qy, float inv_sig2, float (&acc)[4]) {
    const float t = fminf(fmaxf(t0, 0.f), 1.f);
    const float k = coef * 4.f * d2 * g * inv_sig2;        // coef * dg/dd2 * (-2)
    const float ka = k * (1.f - t), kb = k * t;
    acc[0] = fmaf(ka, qx, acc[0]); acc[1] = fmaf(ka, qy, acc[1]);
    acc[2] = fmaf(kb, qx, acc[2]); acc[3] = fmaf(kb, qy, acc[3]);
}

// grid = (chunks, L): each CTA reduces a slice of one line's frame
__global__ void __launch_bounds__(256) dense_bwd_kernel(const float* __restrict__ lines, int L, int ts0, int ts1, float sig2, float inv_sig2,
                                                        const float* __restrict__ g_out, float* __restrict__ d_lines) {
    const int l = blockIdx.y;
    const size_t frame = (size_t)ts0 * ts1;
    const float4 e = __ldg(reinterpret_cast<const float4*>(lines) + l);
    const Seg s = {e.x * (float)ts0, e.y * (float)ts1, e.z * (float)ts0, e.w * (float)ts1};
    const float* go = g_out + (size_t)l * frame;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < frame; t += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(t / ts0), c = (int)(t - (size_t)r * ts0);
        float t0, qx, qy;
        const float d2 = seg_dist2((float)c, (float)r, s, t0, qx, qy);
        const float g = line_g(d2, sig2);
        if (g != 0.f) seg_accum(go[t], g, d2, t0, qx, qy, inv_sig2, acc);
    }
    __shared__ float red[4][8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        acc[k] = warp_sum(acc[k]);
        if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = acc[k];
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        float v = 0.f;
        for (int i = 0; i < 8; ++i) v += red[threadIdx.x][i];
        atomicAdd(&d_lines[4 * l + threadIdx.x], v * ((threadIdx.x & 1) ? (float)ts1 : (float)ts0));
    }
}

struct ReduceParams {
    const float* lines;
    int L, ts0, ts1;
    float sig2, inv_sig2, cut;
    float* out_sum; float* out_softor;
    const float* g_sum; const float* g_softor;
    float* d_lines;
};

__device__ __forceinline__ void stage_lines(Seg* seg_s, const ReduceParams& q, int base, int n) {
    __syncthreads();
    if ((int)threadIdx.x < n) {
        const float4 e = __ldg(reinterpret_cast<const float4*>(q.lines) + base + threadIdx.x);
        seg_s[threadIdx.x] = {e.x * (float)q.ts0, e.y * (float)q.ts1, e.z * (float)q.ts0, e.w * (float)q.ts1};
    }
    __syncthreads();
}

template <bool SUM, bool SOFTOR>
__global__ void __launch_bounds__(CTA) reduce_fwd_kernel(ReduceParams q) {
    __shared__ Seg seg_s[CHUNK];
    const int tiles_x = (q.ts0 + TCOLS - 1) / TCOLS;
    const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c = tx * TCOLS + lane, r0 = ty * TROWS + warp * WROWS;
    const float cf = (float)c, x0 = (float)(tx * TCOLS), y0 = (float)r0;
    float acc_s[WROWS], acc_p[WROWS];
#pragma unroll
    for (int i = 0; i < WROWS; ++i) { acc_s[i] = 0.f; acc_p[i] = 1.f; }
    for (int base = 0; base < q.L; base += CHUNK) {
        const int n = min(CHUNK, q.L - base);
        stage_lines(seg_s, q, base, n);
        for (int k = 0; k < n; ++k) {
            const Seg s = seg_s[k];
            if (!seg_near_block(s, x0, y0, (float)TCOLS, (float)WROWS, q.cut)) continue;      // warp-uniform
#pragma unroll
            for (int i = 0; i < WROWS; ++i) {
                float t0, qx, qy;
                const float g = line_g(seg_dist2(cf, y0 + (float)i, s, t0, qx, qy), q.sig2);
                if (SUM) acc_s[i] += g;
                if (SOFTOR) acc_p[i] *= 1.f - g;
            }
        }
    }
    if (c < q.ts0) {
#pragma unroll
        for (int i = 0; i < WROWS; ++i) {
            if (r0 + i < q.ts1) {
                if (SUM) q.out_sum[(size_t)(r0 + i) * q.ts0 + c] = acc_s[i];
                if (SOFTOR) q.out_softor[(size_t)(r0 + i) * q.ts0 + c] = 1.f - acc_p[i];
            }
        }
    }
}

template <bool SUM, bool SOFTOR>
__global__ void __launch_bounds__(CTA) reduce_bwd_kernel(ReduceParams q) {
    __shared__ Seg seg_s[CHUNK];
    __shared__ float dl_s[CHUNK][4];
    const int tiles_x = (q.ts0 + TCOLS - 1) / TCOLS;
    const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c = tx * TCOLS + lane, r0 = ty * TROWS + warp * WROWS;
    const float cf = (float)c, x0 = (float)(tx * TCOLS), y0 = (float)r0;
    float gs[WROWS], go[WROWS], prod[WROWS];
    uint32_t z1 = 0, z2 = 0;                   // bit i: >= 1 / >= 2 exact-zero factors (texel on a line) at row i
#pragma unroll
    for (int i = 0; i < WROWS; ++i) {
        const bool in = c < q.ts0 && r0 + i < q.ts1;
        gs[i] = (SUM && in) ? __ldg(q.g_sum + (size_t)(r0 + i) * q.ts0 + c) : 0.f;
        go[i] = (SOFTOR && in) ? __ldg(q.g_softor + (size_t)(r0 + i) * q.ts0 + c) : 0.f;
        prod[i] = 1.f;
    }
    if (SOFTOR) {                              // pass 1: product of the non-zero (1 - g) factors per texel
        for (int base = 0; base < q.L; base += CHUNK) {
            const int n = min(CHUNK, q.L - base);
            stage_lines(seg_s, q, base, n);
            for (int k = 0; k < n; ++k) {
                const Seg s = seg_s[k];
                if (!seg_near_block(s, x0, y0, (float)TCOLS, (float)WROWS, q.cut)) continue;
#pragma unroll
                for (int i = 0; i < WROWS; ++i) {
                    float t0, qx, qy;
                    const float om = 1.f - line_g(seg_dist2(cf, y0 + (float)i, s, t0, qx, qy), q.sig2);
                    if (om == 0.f) { z2 |= z1 & (1u << i); z1 |= 1u << i; }
                    else prod[i] *= om;
                }
            }
        }
    }
    for (int base = 0; base < q.L; base += CHUNK) {          // pass 2
        const int n = min(CHUNK, q.L - base);
        stage_lines(seg_s, q, base, n);
        if ((int)threadIdx.x < n) { dl_s[threadIdx.x][0] = 0.f; dl_s[threadIdx.x][1] = 0.f; dl_s[threadIdx.x][2] = 0.f; dl_s[threadIdx.x][3] = 0.f; }
        __syncthreads();
        for (int k = 0; k < n; ++k) {
            const Seg s = seg_s[k];
            if (!seg_near_block(s, x0, y0, (float)TCOLS, (float)WROWS, q.cut)) continue;
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int i = 0; i < WROWS; ++i) {
                float t0, qx, qy;
                const float d2 = seg_dist2(cf, y0 + (float)i, s, t0, qx, qy);
                const float g = line_g(d2, q.sig2);
                float coef = SUM ? gs[i] : 0.f;
                if (SOFTOR) {
                    const float om = 1.f - g;
                    float excl;                               // prod_{m != n} (1 - g_m), as torch.prod's backward
                    if (!(z1 & (1u << i))) excl = __fdividef(prod[i], om);
                    else excl = (om == 0.f && !(z2 & (1u << i))) ? prod[i] : 0.f;
                    coef = fmaf(go[i], excl, coef);
                }
                if (g != 0.f) seg_accum(coef, g, d2, t0, qx, qy, q.inv_sig2, acc);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                acc[j] = warp_sum(acc[j]);
                if (lane == 0 && acc[j] != 0.f) atomicAdd(&dl_s[k][j], acc[j]);
            }
        }
        __syncthreads();
        for (int e = threadIdx.x; e < 4 * n; e += CTA) {      // 4 * CHUNK components, more than one per thread
            const int k = e >> 2, j = e & 3;
            const float v = dl_s[k][j] * ((j & 1) ? (float)q.ts1 : (float)q.ts0);
            if (v != 0.f) atomicAdd(&q.d_lines[4 * (base + k) + j], v);
        }
    }
}

// ---- depth ---------------------------------------------------------------------------------------------------------
// g at the texel nearest to P inside the frame = the maximum of the dense splat over the frame (g decreases with |dc| and |dr|)
__device__ __forceinline__ float depth_gmax(float p0, float p1, int ts0, int ts1, float sigma, float rcp_sigma, float& dcm, float& drm) {
    const float cm = fminf(fmaxf(rintf(p0), 0.f), (float)(ts0 - 1)), rm = fminf(fmaxf(rintf(p1), 0.f), (float)(ts1 - 1));
    dcm = cm - p0; drm = rm - p1;
    const float d2 = __fadd_rn(__fmul_rn(dcm, dcm), __fmul_rn(drm, drm));
    const float u = div_by(d2, sigma, rcp_sigma);
    const float w = __fmul_rn(u, u);
    return w > 87.f ? 0.f : exp_neg(w);
}

// out[n,r,c] = g / max_frame(g) * depth[n]   (rasterization.py:66-104)
__global__ void __launch_bounds__(256) depth_fwd_kernel(const float* __restrict__ pts, const float* __restrict__ depth, int N, int ts0, int ts1,
                                                        float sigma, float rcp_sigma, float* __restrict__ out) {
    const size_t frame = (size_t)ts0 * ts1, total = frame * N;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int n = (int)(i / frame);
        const size_t t = i - (size_t)n * frame;
        const int r = (int)(t / ts0), c = (int)(t - (size_t)r * ts0);
        const float p0 = pts[2 * n] * (float)ts0, p1 = pts[2 * n + 1] * (float)ts1;
        const float dx = (float)c - p0, dy = (float)r - p1;
        const float d2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
        const float u = div_by(d2, sigma, rcp_sigma);
        const float w = __fmul_rn(u, u);
        const float g = w > 87.f ? 0.f : exp_neg(w);
        float a, b;
        const float gm = depth_gmax(p0, p1, ts0, ts1, sigma, rcp_sigma, a, b);
        out[i] = __fmul_rn(__fdiv_rn(g, gm), depth[n]);
    }
}

// soft-OR over the points of the normalised, depth-scaled splat: 1 - prod_n (1 - depth_n g_n / gmax_n)   (rasterization.py:538-549)
__global__ void __launch_bounds__(256) depth_softor_kernel(const float* __restrict__ pts, const float* __restrict__ depth, int N, int ts0, int ts1,
                                                           float sigma, float rcp_sigma, float* __restrict__ out) {
    extern __shared__ float4 rec_s[];          // p0, p1, depth / gmax (as two factors: depth, gmax)
    const size_t frame = (size_t)ts0 * ts1;
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int r = (int)(t / ts0), c = (int)(t - (size_t)r * ts0);
    float p = 1.f;
    for (int base = 0; base < N; base += 256) {
        const int n = min(256, N - base);
        __syncthreads();
        if ((int)threadIdx.x < n) {
            const float p0 = pts[2 * (base + threadIdx.x)] * (float)ts0, p1 = pts[2 * (base + threadIdx.x) + 1] * (float)ts1;
            float a, b;
            rec_s[threadIdx.x] = make_float4(p0, p1, depth[base + threadIdx.x], depth_gmax(p0, p1, ts0, ts1, sigma, rcp_sigma, a, b));
        }
        __syncthreads();
        if (t < frame) {
            for (int k = 0; k < n; ++k) {
                const float4 e = rec_s[k];
                const float dx = (float)c - e.x, dy = (float)r - e.y;
                const float d2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
                const float u = div_by(d2, sigma, rcp_sigma);
                const float w = __fmul_rn(u, u);
                const float g = w > 87.f ? 0.f : exp_neg(w);
                p *= 1.f - __fmul_rn(__fdiv_rn(g, e.w), e.z);
            }
        }
    }
    if (t < frame) out[t] = 1.f - p;
}

// backward of depth_fwd_kernel: with A = depth / gmax, out = A g:
//   d/dp   = A sum go dg/dp  -  (sum go g) A / gmax * dgmax/dp        d/d depth = (sum go g) / gmax
// grid = (chunks, N); partial sums (S0, S1 = sum go dg/dp, Sg = sum go g) land in `part` [N,3] through atomics, then
// depth_bwd_finish combines them.
__global__ void __launch_bounds__(256) depth_bwd_kernel(const float* __restrict__ pts, int N, int ts0, int ts1, float sigma, float rcp_sigma,
                                                        const float* __restrict__ g_out, float* __restrict__ part) {
    const int n = blockIdx.y;
    const size_t frame = (size_t)ts0 * ts1;
    const float p0 = pts[2 * n] * (float)ts0, p1 = pts[2 * n + 1] * (float)ts1;
    const float* go = g_out + (size_t)n * frame;
    float a0 = 0.f, a1 = 0.f, ag = 0.f;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < frame; t += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(t / ts0), c = (int)(t - (size_t)r * ts0);
        const float dx = (float)c - p0, dy = (float)r - p1;
        const float u = (dx * dx + dy * dy) * rcp_sigma;
        const float w = u * u;
        if (w <= 87.f) {
            const float g = exp_neg(w), v = go[t];
            const float qg = v * g * u;
            a0 = fmaf(qg, dx, a0); a1 = fmaf(qg, dy, a1); ag = fmaf(v, g, ag);
        }
    }
    __shared__ float red[3][8];
    a0 = warp_sum(a0); a1 = warp_sum(a1); ag = warp_sum(ag);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a0; red[1][threadIdx.x >> 5] = a1; red[2][threadIdx.x >> 5] = ag; }
    __syncthreads();
    if (threadIdx.x < 3) {
        float s = 0.f;
        for (int i = 0; i < 8; ++i) s += red[threadIdx.x][i];
        atomicAdd(&part[3 * n + threadIdx.x], s);
    }
}
__global__ void depth_bwd_finish(const float* __restrict__ pts, const float* __restrict__ depth, int N, int ts0, int ts1, float sigma,
                                 float rcp_sigma, const float* __restrict__ part, float* __restrict__ d_pts, float* __restrict__ d_depth) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float p0 = pts[2 * n] * (float)ts0, p1 = pts[2 * n + 1] * (float)ts1;
    float dcm, drm;
    const float gm = depth_gmax(p0, p1, ts0, ts1, sigma, rcp_sigma, dcm, drm);
    const float A = depth[n] / gm;
    const float um = (dcm * dcm + drm * drm) * rcp_sigma;
    // dg/dP = 4 g u (c - P) / sigma (texture units); dgmax/dP likewise at the nearest texel
    const float k = 4.f * rcp_sigma;
    const float S0 = part[3 * n] * k, S1 = part[3 * n + 1] * k, Sg = part[3 * n + 2];
    const float dm0 = k * gm * um * dcm, dm1 = k * gm * um * drm;
    if (d_pts) {
        d_pts[2 * n] = (A * S0 - Sg * A / gm * dm0) * (float)ts0;
        d_pts[2 * n + 1] = (A * S1 - Sg * A / gm * dm1) * (float)ts1;
    }
    if (d_depth) d_depth[n] = Sg / gm;
}

}  // namespace lines
}  // namespace ffb

using namespace ffb;
using namespace ffb::lines;

static int lines_args(const float* lines, int32_t L, int32_t ts0, int32_t ts1, float sigma, const char* who) {
    if (!lines || L <= 0 || ts0 <= 0 || ts1 <= 0 || !(sigma > 0.f)) {
        snprintf(last_error_buf(), 256, "%s: bad argument", who);
        return FFB_E_ARG;
    }
    if ((reinterpret_cast<uintptr_t>(lines) & 15) != 0) {
        snprintf(last_error_buf(), 256, "%s: lines must be 16-byte aligned", who);
        return FFB_E_ARG;
    }
    return 0;
}

extern "C" int ffb_lines_dense_fwd(const float* lines, int32_t L, int32_t ts0, int32_t ts1, float sigma, float* out, void* stream) {
    if (int rc = lines_args(lines, L, ts0, ts1, sigma, "lines_dense_fwd")) return rc;
    if (!out) return fail_arg(FFB_E_ARG, "lines_dense_fwd: null output");
    const size_t total = (size_t)L * ts0 * ts1;
    size_t blocks = (total + 255) / 256;
    if (blocks > (size_t)kNumSMs * 32) blocks = (size_t)kNumSMs * 32;
    dense_fwd_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(lines, L, ts0, ts1, sigma * sigma, out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_lines_dense_bwd(const float* lines, int32_t L, int32_t ts0, int32_t ts1, float sigma, const float* g_out,
                                   float* d_lines, void* stream) {
    if (int rc = lines_args(lines, L, ts0, ts1, sigma, "lines_dense_bwd")) return rc;
    if (!g_out || !d_lines) return fail_arg(FFB_E_ARG, "lines_dense_bwd: null pointer");
    if (L > 65535) return fail_arg(FFB_E_LIMIT, "lines_dense_bwd: L > 65535");
    cudaStream_t st = as_stream(stream);
    FFB_CUDA(cudaMemsetAsync(d_lines, 0, (size_t)L * 4 * sizeof(float), st));
    const size_t frame = (size_t)ts0 * ts1;
    unsigned chunks = (unsigned)((frame + 256 * 16 - 1) / (256 * 16));
    if (chunks > 64) chunks = 64;
    if (chunks < 1) chunks = 1;
    dense_bwd_kernel<<<dim3(chunks, L), 256, 0, st>>>(lines, L, ts0, ts1, sigma * sigma, 1.0f / (sigma * sigma), g_out, d_lines);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

static void fill_reduce(ReduceParams& q, const float* lines, int32_t L, int32_t ts0, int32_t ts1, float sigma) {
    q.lines = lines; q.L = L; q.ts0 = ts0; q.ts1 = ts1;
    q.sig2 = sigma * sigma; q.inv_sig2 = 1.0f / (sigma * sigma);
    q.cut = sqrtf(sigma * sqrtf(88.f) * 1.01f);            // beyond it (d2^2 / sigma^2 > 87) g underflows to 0
    q.out_sum = nullptr; q.out_softor = nullptr; q.g_sum = nullptr; q.g_softor = nullptr; q.d_lines = nullptr;
}

extern "C" int ffb_lines_reduce_fwd(const float* lines, int32_t L, int32_t ts0, int32_t ts1, float sigma, float* out_sum,
                                    float* out_softor, void* stream) {
    if (int rc = lines_args(lines, L, ts0, ts1, sigma, "lines_reduce_fwd")) return rc;
    if (!out_sum && !out_softor) return fail_arg(FFB_E_ARG, "lines_reduce_fwd: no output requested");
    ReduceParams q;
    fill_reduce(q, lines, L, ts0, ts1, sigma);
    q.out_sum = out_sum; q.out_softor = out_softor;
    const unsigned grid = (unsigned)(((ts0 + TCOLS - 1) / TCOLS) * ((ts1 + TROWS - 1) / TROWS));
    cudaStream_t st = as_stream(stream);
    if (out_sum && out_softor) reduce_fwd_kernel<true, true><<<grid, CTA, 0, st>>>(q);
    else if (out_sum) reduce_fwd_kernel<true, false><<<grid, CTA, 0, st>>>(q);
    else reduce_fwd_kernel<false, true><<<grid, CTA, 0, st>>>(q);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_lines_reduce_bwd(const float* lines, int32_t L, int32_t ts0, int32_t ts1, float sigma, const float* g_sum,
                                    const float* g_softor, float* d_lines, void* stream) {
    if (int rc = lines_args(lines, L, ts0, ts1, sigma, "lines_reduce_bwd")) return rc;
    if (!d_lines) return fail_arg(FFB_E_ARG, "lines_reduce_bwd: null pointer");
    if (!g_sum && !g_softor) return fail_arg(FFB_E_ARG, "lines_reduce_bwd: no upstream gradient");
    ReduceParams q;
    fill_reduce(q, lines, L, ts0, ts1, sigma);
    q.g_sum = g_sum; q.g_softor = g_softor; q.d_lines = d_lines;
    cudaStream_t st = as_stream(stream);
    FFB_CUDA(cudaMemsetAsync(d_lines, 0, (size_t)L * 4 * sizeof(float), st));
    const unsigned grid = (unsigned)(((ts0 + TCOLS - 1) / TCOLS) * ((ts1 + TROWS - 1) / TROWS));
    if (g_sum && g_softor) reduce_bwd_kernel<true, true><<<grid, CTA, 0, st>>>(q);
    else if (g_sum) reduce_bwd_kernel<true, false><<<grid, CTA, 0, st>>>(q);
    else reduce_bwd_kernel<false, true><<<grid, CTA, 0, st>>>(q);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_depth_dense_fwd(const float* pts, const float* depth, int32_t N, int32_t ts0, int32_t ts1, float sigma, float* out,
                                   void* stream) {
    if (!pts || !depth || !out || N <= 0 || ts0 <= 0 || ts1 <= 0 || !(sigma > 0.f)) return fail_arg(FFB_E_ARG, "depth_dense_fwd: bad argument");
    const size_t total = (size_t)N * ts0 * ts1;
    size_t blocks = (total + 255) / 256;
    if (blocks > (size_t)kNumSMs * 32) blocks = (size_t)kNumSMs * 32;
    depth_fwd_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(pts, depth, N, ts0, ts1, sigma, 1.0f / sigma, out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_depth_softor_fwd(const float* pts, const float* depth, int32_t N, int32_t ts0, int32_t ts1, float sigma, float* out,
                                    void* stream) {
    if (!pts || !depth || !out || N <= 0 || ts0 <= 0 || ts1 <= 0 || !(sigma > 0.f)) return fail_arg(FFB_E_ARG, "depth_softor_fwd: bad argument");
    const size_t frame = (size_t)ts0 * ts1;
    depth_softor_kernel<<<(unsigned)((frame + 255) / 256), 256, 256 * sizeof(float4), as_stream(stream)>>>(pts, depth, N, ts0, ts1, sigma,
                                                                                                          1.0f / sigma, out);
    FFB_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int ffb_depth_dense_bwd(const float* pts, const float* depth, int32_t N, int32_t ts0, int32_t ts1, float sigma,
                                   const float* g_out, float* scratch, float* d_pts, float* d_depth, void* stream) {
    if (!pts || !depth || !g_out || !scratch || N <= 0 || ts0 <= 0 || ts1 <= 0 || !(sigma > 0.f))
        return fail_arg(FFB_E_ARG, "depth_dense_bwd: bad argument");
    if (N > 65535) return fail_arg(FFB_E_LIMIT, "depth_dense_bwd: N > 65535");
    cudaStream_t st = as_stream(stream);
    FFB_CUDA(cudaMemsetAsync(scratch, 0, (size_t)N * 3 * sizeof(float), st));
    const size_t frame = (size_t)ts0 * ts1;
    unsigned chunks = (unsigned)((frame + 256 * 16 - 1) / (256 * 16));
    if (chunks > 64) chunks = 64;
    if (chunks < 1) chunks = 1;
    depth_bwd_kernel<<<dim3(chunks, N), 256, 0, st>>>(pts, N, ts0, ts1, sigma, 1.0f / sigma, g_out, scratch);
    FFB_CUDA(cudaGetLastError());
    depth_bwd_finish<<<(N + 127) / 128, 128, 0, st>>>(pts, depth, N, ts0, ts1, sigma, 1.0f / sigma, scratch, d_pts, d_depth);
    FFB_CUDA(cudaGetLastError());
    return 0;
}
