// Image-space post-processing for sm_100a: separable Gaussian blur (reflect border) fused with white
// noise + clip, per-frame Bernoulli gates.
//
// Replaces (reference paths relative to the Fireflies tree):
//   fireflies/postprocessing/gauss_blur.py:18-28   GaussianBlur.post_process -> kornia.filters.gaussian_blur2d
//   fireflies/postprocessing/white_noise.py:16-20  WhiteNoise.post_process
//   fireflies/postprocessing/base.py:10-14, postprocessor.py:14-19  (gates are drawn by the caller)
//
// HBM-bound stencil.  Production kernel (blur_sw_kernel, the kernel sizes the reference uses: 3, 5, 11): each CTA
// produces a 128-column tile, 8 or 16 rows per warp.  The input tile + halo is fetched by ONE TMA tensor load
// (cp.async.bulk.tensor.3d) into shared memory; out-of-image halo cells arrive as zeros and edge tiles patch them
// with the reflected in-tile cells (kornia border_type="reflect", no edge repeat), so the inner loops carry no
// index arithmetic.  (Measured on B200: the innermost TMA start coordinate must be a multiple of 16 bytes --
// x = -1 raises 'illegal instruction', x = -4 works, any y works -- so the left halo is padded to 4 texels.)
// A lane owns 4 columns: per input row it reads aligned 128-bit words, forms the 4 horizontal sums with
// compile-time taps, pushes them into a register sliding window of KY rows and emits one output row
// (vertical taps, noise / clip in registers, one 128-bit store).  No intermediate shared-memory pass.
// Traffic: 4 B read (+ halo re-reads served by L2) + 4 B written per texel.
// Other odd kernel sizes up to 15 take the generic kernel (blur_kernel: smem->smem horizontal, smem->register vertical).
// The blur's adjoint (ffb_blur_bwd, what autograd needs to carry a gradient through the blur): blur_bwd_sw_kernel on the
// sliding-window kernel's inputs, blur_bwd_kernel (plain loads) on every other input the forward accepts.
#include <cuda.h>

#include "ffb_common.cuh"
#include "ffb_tma.cuh"

namespace ffb {
namespace post {

constexpr int TW = 128, TH = 32, THREADS = 256, KMAX = 15;

struct PostParams {
    int B, H, W;
    int kx, ky, hx, hy;          // taps and left/top halo (k/2)
    int padl;                    // left halo rounded up to 4 texels: TMA needs a 16-byte aligned inner start coordinate
    int boxw, boxh;              // TMA box (boxw multiple of 4)
    float wx[KMAX], wy[KMAX];
    int noise;
    float mean, stdv;
    uint64_t seed, frame0;
    const float* img;
    const uint8_t* gates;        // [B,2] or null
    const double* noise_inj;     // [B,H,W] or null
    const float* mul;            // [B,H,W] or null: the result is multiplied texel-wise (silhouette: image x blurred mask)
    float* out;
};

__device__ __forceinline__ int reflect(int i, int n) {      // torch 'reflect' padding (pad < n)
    i = i < 0 ? -i : i;
    return i >= n ? 2 * (n - 1) - i : i;
}

// 8 normal variates for a 4-texel quad of two consecutive rows (2 rp, 2 rp + 1) of one frame: one Philox4x32-10 call keyed by
// the seed, counter = (row-pair quad index, global frame index); every 32-bit output feeds one Box-Muller pair (upper 16
// bits: radius, u in (0, 1]; lower 16 bits: angle), so a call yields eight variates -- the integer rounds were two thirds
// of the noise stage's instructions when a call served four.  The 16-bit radius caps |z| at 4.7 (P = 2.6e-6); the stream
// has statistical parity with numpy's only (SURVEY.md 8(c)).  Independent of tiling, batching and rank.
__device__ __forceinline__ void normal8(uint64_t seed, uint64_t frame, uint32_t quadpair, float (&za)[4], float (&zb)[4]) {
    uint32_t r[4];
    Philox::gen(seed, quadpair, 0x4E015E00u, (uint32_t)frame, (uint32_t)(frame >> 32), r);
    // Box-Muller on the special-function unit: lg2, rsqrt, sin, cos (absolute error ~1e-6)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float u0 = ((float)(r[k] >> 16) + 1.0f) * (1.0f / 65536.0f), u1 = (float)(r[k] & 0xffffu) * (1.0f / 65536.0f);
        const float x2 = -1.3862943611198906f * __log2f(u0);                      // -2 ln u
        const float rad = x2 * rsqrtf(fmaxf(x2, 1e-30f));
        float sn, cs;
        __sincosf(6.283185307179586f * u1, &sn, &cs);
        if (k < 2) { za[2 * k] = rad * cs; za[2 * k + 1] = rad * sn; }          // row 2 rp
        else { zb[2 * k - 4] = rad * cs; zb[2 * k - 3] = rad * sn; }            // row 2 rp + 1
    }
}
__device__ __forceinline__ uint32_t quadpair_index(const PostParams& q, int y, int x0) {
    return (uint32_t)((size_t)(y >> 1) * ((size_t)(q.W + 3) / 4) + (size_t)(x0 >> 2));
}

// noise + clip on up to 4 consecutive texels (x0..x0+3 of row y) given their variates -- white_noise.py:17-20
__device__ __forceinline__ void noise_clip4z(const PostParams& q, int b, int y, int x0, float (&v)[4], const float (&z)[4]) {
    if (q.noise_inj) {
        const size_t base = ((size_t)b * q.H + y) * q.W + x0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (x0 + k < q.W) v[k] = (float)((double)v[k] + q.noise_inj[base + k]);    // fp32 image += fp64 draw
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] += fmaf(q.stdv, z[k], q.mean);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = fminf(fmaxf(v[k], 0.f), 1.f);
}
// stateless form: generates the row pair's eight variates and uses this row's four
__device__ __forceinline__ void noise_clip4(const PostParams& q, int b, int y, int x0, float (&v)[4]) {
    float za[4] = {0.f, 0.f, 0.f, 0.f}, zb[4] = {0.f, 0.f, 0.f, 0.f};
    if (!q.noise_inj) normal8(q.seed, q.frame0 + (uint64_t)b, quadpair_index(q, y, x0), za, zb);
    if (y & 1) noise_clip4z(q, b, y, x0, v, zb);
    else noise_clip4z(q, b, y, x0, v, za);
}

__device__ __forceinline__ void store4(const PostParams& q, int b, int y, int x0, const float (&vin)[4]) {
    const size_t off = ((size_t)b * q.H + y) * q.W + x0;
    float* o = q.out + off;
    float v[4] = {vin[0], vin[1], vin[2], vin[3]};
    const bool vec = x0 + 4 <= q.W && (q.W & 3) == 0;
    if (q.mul) {                                             // warp-uniform
        if (vec) {
            const float4 m = __ldg(reinterpret_cast<const float4*>(q.mul + off));
            v[0] *= m.x; v[1] *= m.y; v[2] *= m.z; v[3] *= m.w;
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (x0 + k < q.W) v[k] *= __ldg(q.mul + off + k);
        }
    }
    if (vec) *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
    else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (x0 + k < q.W) o[k] = v[k];
    }
}

// mbarrier / TMA PTX helpers: ffb_tma.cuh (shared with the splat kernels)
using tma::mbar_init;
using tma::mbar_expect_tx;
using tma::mbar_wait;
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int x, int y, int z) {
    tma::load_3d(dst, map, bar, x, y, z);
}

// Blur (+ optional noise/clip) of one 128x32 tile.  USE_TMA = false is the fallback for W % 4 != 0 (TMA
// needs 16-byte global strides): the same arithmetic, tile filled with plain loads.
template <bool USE_TMA>
__global__ void __launch_bounds__(THREADS) blur_kernel(const __grid_constant__ CUtensorMap tmap, const PostParams q) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* in_s = reinterpret_cast<float*>(smem_raw);                  // [boxh][boxw]
    float* mid_s = in_s + q.boxh * q.boxw;                              // [boxh][TW]
    __shared__ __align__(8) uint64_t bar;
    const int tiles_x = (q.W + TW - 1) / TW;
    const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x, b = blockIdx.y;
    const int x0 = tx * TW, y0 = ty * TH;
    const int tid = threadIdx.x;
    const bool do_blur = q.gates ? q.gates[b * 2] != 0 : true;
    const bool do_noise = q.noise && (q.gates ? q.gates[b * 2 + 1] != 0 : true);

    if (!do_blur) {      // gate off: copy (PostProcessor copies once) [+ noise]
        for (int i = tid; i < (TW / 4) * TH; i += THREADS) {
            const int y = y0 + i / (TW / 4), x = x0 + (i % (TW / 4)) * 4;
            if (y >= q.H || x >= q.W) continue;
            float v[4];
            const float* s = q.img + ((size_t)b * q.H + y) * q.W + x;
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = x + k < q.W ? __ldg(s + k) : 0.f;
            if (do_noise) noise_clip4(q, b, y, x, v);
            store4(q, b, y, x, v);
        }
        return;
    }

    // ---- stage input tile + halo ----
    const int gx0 = x0 - q.padl, gy0 = y0 - q.hy;
    if (USE_TMA) {
        if (tid == 0) {
            mbar_init(&bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (tid == 0) {
            mbar_expect_tx(&bar, (uint32_t)(q.boxw * q.boxh * sizeof(float)));
            tma_load_3d(in_s, &tmap, &bar, gx0, gy0, b);
        }
        mbar_wait(&bar, 0);
    } else {
        for (int i = tid; i < q.boxw * q.boxh; i += THREADS) {
            const int ly = i / q.boxw, lx = i - ly * q.boxw;
            const int gy = gy0 + ly, gx = gx0 + lx;
            in_s[i] = (gy >= 0 && gy < q.H && gx >= 0 && gx < q.W) ? __ldg(q.img + ((size_t)b * q.H + gy) * q.W + gx) : 0.f;
        }
        __syncthreads();
    }

    // ---- horizontal pass: mid[j][i] = sum_t wx[t] * in[j][reflect(x0 + i + t - hx)] ----
    const bool edge_x = (x0 == 0) || (x0 + TW + (q.kx - 1 - q.hx) > q.W);
    const int rows_used = q.boxh;
    for (int idx = tid; idx < rows_used * TW; idx += THREADS) {
        const int j = idx / TW, i = idx - j * TW;
        const int gy = gy0 + j;
        float acc = 0.f;
        if (gy >= 0 && gy < q.H && x0 + i < q.W) {
            const float* row = in_s + j * q.boxw;
            if (!edge_x) {
                const float* r2 = row + i + (q.padl - q.hx);
                for (int t = 0; t < q.kx; ++t) acc = fmaf(q.wx[t], r2[t], acc);
            } else {
                for (int t = 0; t < q.kx; ++t) acc = fmaf(q.wx[t], row[reflect(x0 + i + t - q.hx, q.W) - gx0], acc);
            }
        }
        mid_s[j * TW + i] = acc;
    }
    __syncthreads();

    // ---- vertical pass + epilogue: each thread 4 consecutive columns of 4 rows ----
    const int cg = tid & 31, r_base = tid >> 5;
    const int x = x0 + cg * 4;
#pragma unroll
    for (int k = 0; k < TH / 8; ++k) {
        const int r = r_base + k * 8, y = y0 + r;
        if (y >= q.H || x >= q.W) continue;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        for (int t = 0; t < q.ky; ++t) {
            const int j = reflect(y + t - q.hy, q.H) - gy0;
            const float4 m = *reinterpret_cast<const float4*>(mid_s + j * TW + cg * 4);
            v[0] = fmaf(q.wy[t], m.x, v[0]); v[1] = fmaf(q.wy[t], m.y, v[1]);
            v[2] = fmaf(q.wy[t], m.z, v[2]); v[3] = fmaf(q.wy[t], m.w, v[3]);
        }
        if (do_noise) noise_clip4(q, b, y, x, v);
        store4(q, b, y, x, v);
    }
}


// ---- sliding-window blur ----------------------------------------------------------------------------------------------
constexpr int SW_TW = 128;                 // tile width: 32 lanes x 4 columns
template <int K> struct SwCfg {
    static constexpr int H = K / 2;                      // taps each side
    static constexpr int PADL = (H + 3) & ~3;            // left / right halo rounded to 4 texels (TMA alignment, aligned LDS.128)
    static constexpr int NQ = PADL / 4;                  // extra 128-bit words each side
    static constexpr int RW = K <= 5 ? 8 : 16;           // output rows per warp
    static constexpr int TH = 8 * RW;                    // tile height (8 warps)
    static constexpr int BOXW = SW_TW + 2 * PADL;
    static constexpr int BOXH = TH + K - 1;
};

// NOISE / MUL: the launch has a noise stage / a texel-wise multiplier; the plain blur instantiation carries neither the
// variate registers nor the multiplier load
template <int KX, int KY, bool NOISE, bool MUL>
__global__ void __launch_bounds__(THREADS) blur_sw_kernel(const __grid_constant__ CUtensorMap tmap, const PostParams qin) {
    PostParams q = qin;
    if (!MUL) q.mul = nullptr;
    typedef SwCfg<KX> CX;
    typedef SwCfg<KY> CY;
    constexpr int BOXW = CX::BOXW, BOXH = CY::BOXH, TH2 = CY::TH, RW = CY::RW;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* in_s = reinterpret_cast<float*>(smem_raw);                  // [BOXH][BOXW]
    __shared__ __align__(8) uint64_t bar;
    const int tiles_x = (q.W + SW_TW - 1) / SW_TW;
    const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x, b = blockIdx.y;
    const int x0 = tx * SW_TW, y0 = ty * TH2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool do_blur = q.gates ? q.gates[b * 2] != 0 : true;
    const bool do_noise = NOISE && q.noise && (q.gates ? q.gates[b * 2 + 1] != 0 : true);

    if (!do_blur) {      // gate off: copy (PostProcessor copies once) [+ noise]
        for (int i = tid; i < (SW_TW / 4) * TH2; i += THREADS) {
            const int y = y0 + i / (SW_TW / 4), x = x0 + (i % (SW_TW / 4)) * 4;
            if (y >= q.H || x >= q.W) continue;
            float v[4];
            const float4 a = __ldg(reinterpret_cast<const float4*>(q.img + ((size_t)b * q.H + y) * q.W + x));   // W % 4 == 0 on this path
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
            if (do_noise) noise_clip4(q, b, y, x, v);
            store4(q, b, y, x, v);
        }
        return;
    }

    // ---- stage input tile + halo (one TMA load), patch the reflect border on edge tiles ----
    const int gx0 = x0 - CX::PADL, gy0 = y0 - CY::H;
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(&bar, (uint32_t)(BOXW * BOXH * sizeof(float)));
        tma_load_3d(in_s, &tmap, &bar, gx0, gy0, b);
    }
    mbar_wait(&bar, 0);
    if (gx0 < 0 || gy0 < 0 || gx0 + BOXW > q.W || gy0 + BOXH > q.H) {
        for (int i = tid; i < BOXW * BOXH; i += THREADS) {
            const int ly = i / BOXW, lx = i - ly * BOXW;
            const int gy = gy0 + ly, gx = gx0 + lx;
            if (gy < 0 || gy >= q.H || gx < 0 || gx >= q.W) {
                // rows / columns beyond the far image edge by more than the halo are never used: clamp keeps the index in the box
                const int sy = min(max(reflect(gy, q.H) - gy0, 0), BOXH - 1), sx = min(max(reflect(gx, q.W) - gx0, 0), BOXW - 1);
                const int ry = reflect(gy, q.H), rx = reflect(gx, q.W);
                const bool ok = ry >= gy0 && ry < gy0 + BOXH && rx >= gx0 && rx < gx0 + BOXW && ry >= 0 && ry < q.H && rx >= 0 && rx < q.W;
                in_s[i] = ok ? in_s[sy * BOXW + sx] : 0.f;
            }
        }
        __syncthreads();
    }

    // ---- per lane: 4 columns, sliding window over the rows of this warp ----
    float wx[KX], wy[KY];
#pragma unroll
    for (int t = 0; t < KX; ++t) wx[t] = q.wx[t];
#pragma unroll
    for (int t = 0; t < KY; ++t) wy[t] = q.wy[t];
    const int x = x0 + 4 * lane;
    const float* colp = in_s + 4 * lane;                     // first 128-bit word of this lane's window (PADL texels left of its columns)
    float win[KY][4];
    float za[4] = {0.f, 0.f, 0.f, 0.f}, zb[4] = {0.f, 0.f, 0.f, 0.f};   // the row pair's variates: generated on even rows, zb kept for the odd row
#pragma unroll
    for (int rr = 0; rr < RW + KY - 1; ++rr) {
        const float* rowp = colp + (warp * RW + rr) * BOXW;
        float v[4 * (1 + 2 * CX::NQ)];
#pragma unroll
        for (int w4 = 0; w4 < 1 + 2 * CX::NQ; ++w4) {
            const float4 a = *reinterpret_cast<const float4*>(rowp + 4 * w4);
            v[4 * w4] = a.x; v[4 * w4 + 1] = a.y; v[4 * w4 + 2] = a.z; v[4 * w4 + 3] = a.w;
        }
        float hsum[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float acc = 0.f;
#pragma unroll
            for (int t = 0; t < KX; ++t) acc = fmaf(wx[t], v[CX::PADL - CX::H + j + t], acc);
            hsum[j] = acc;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) win[rr % KY][j] = hsum[j];
        if (rr >= KY - 1) {
            const int y = y0 + warp * RW + rr - (KY - 1);
            float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int t = 0; t < KY; ++t)
#pragma unroll
                for (int j = 0; j < 4; ++j) o[j] = fmaf(wy[t], win[(rr - (KY - 1) + t) % KY][j], o[j]);
            if (y < q.H && x < q.W) {
                if (do_noise) {
                    // y0 and warp * RW are even and KY is odd: the parity of y is the parity of rr, known at compile time
                    if (((rr - (KY - 1)) & 1) == 0) {
                        if (!q.noise_inj) normal8(q.seed, q.frame0 + (uint64_t)b, quadpair_index(q, y, x), za, zb);
                        noise_clip4z(q, b, y, x, o, za);
                    } else {
                        noise_clip4z(q, b, y, x, o, zb);
                    }
                }
                store4(q, b, y, x, o);
            }
        }
    }
}

template <int KX, int KY>
static int launch_blur_sw(const CUtensorMap& tmap, const PostParams& q, cudaStream_t st) {
    typedef SwCfg<KX> CX;
    typedef SwCfg<KY> CY;
    const size_t smem = (size_t)CX::BOXW * CY::BOXH * sizeof(float);
    const unsigned tiles = (unsigned)(((q.W + SW_TW - 1) / SW_TW) * ((q.H + CY::TH - 1) / CY::TH));
    const bool noise = q.noise != 0, mul = q.mul != nullptr;
#define FFB_SW(N, M)                                                                                                            \
    do {                                                                                                                       \
        if (smem > 48 * 1024)                                                                                                  \
            FFB_CUDA(cudaFuncSetAttribute(blur_sw_kernel<KX, KY, N, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        blur_sw_kernel<KX, KY, N, M><<<dim3(tiles, q.B), THREADS, smem, st>>>(tmap, q);                                         \
    } while (0)
    if (noise && mul) FFB_SW(true, true);
    else if (noise) FFB_SW(true, false);
    else if (mul) FFB_SW(false, true);
    else FFB_SW(false, false);
#undef FFB_SW
    FFB_CUDA(cudaGetLastError());
    return 0;
}

// ---- adjoint of the blur (ffb_blur_bwd) -------------------------------------------------------------------------------
// Per axis the forward is y = W P x (P: reflect padding, W: valid correlation).  The taps are bitwise symmetric, so W^T is
// the same correlation: Z = blur of g with g taken as ZERO outside the image, evaluated on the padded domain
// [-h, n-1+h].  P^T then folds Z back onto the image: x_bar[j] = sum of Z over the preimage set of j under the reflection,
// {j} + {-j if 1 <= j <= h} + {2(n-1)-j if n-1-h <= j <= n-2}; in 2-D over the product of the two axes' sets.  Only texels
// within h of a border (the "band") have more than one preimage.
__device__ __forceinline__ bool in_fold_band(int j, int n, int h) { return (j >= 1 && j <= h) || (j >= n - 1 - h && j <= n - 2); }
// preimage u of j: u = 0 is j itself, 1 the reflection at the low border, 2 at the high one; false if it does not exist
__device__ __forceinline__ bool fold_preimage(int u, int j, int n, int h, int& p) {
    if (u == 0) { p = j; return true; }
    if (u == 1) { p = -j; return j >= 1 && j <= h; }
    p = 2 * (n - 1) - j;
    return j >= n - 1 - h && j <= n - 2;
}

// Generic form: any odd sizes <= 15, W % 4 != 0, unaligned pointers.  One thread per texel, plain loads, the preimage
// formula evaluated directly (q.img = g_out, q.out = g_in).
__global__ void __launch_bounds__(THREADS) blur_bwd_kernel(const PostParams q) {
    const size_t plane = (size_t)q.H * q.W, total = plane * q.B;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(i / plane);
        const int j = (int)((i - (size_t)b * plane) / q.W), c = (int)(i - (size_t)b * plane - (size_t)j * q.W);
        const float* g = q.img + (size_t)b * plane;
        float acc = 0.f;
#pragma unroll 1
        for (int u = 0; u < 3; ++u)
#pragma unroll 1
            for (int v = 0; v < 3; ++v) {
                int p, pc;
                if (!fold_preimage(u, j, q.H, q.hy, p) || !fold_preimage(v, c, q.W, q.hx, pc)) continue;
                float z = 0.f;
                for (int s = 0; s < q.ky; ++s) {
                    const int y = p + s - q.hy;
                    float hs = 0.f;
                    if (y >= 0 && y < q.H)
                        for (int t = 0; t < q.kx; ++t) {
                            const int x = pc + t - q.hx;
                            if (x >= 0 && x < q.W) hs = fmaf(q.wx[t], __ldg(g + (size_t)y * q.W + x), hs);
                        }
                    z = fmaf(q.wy[s], hs, z);
                }
                acc += z;
            }
        q.out[i] = acc;
    }
}

// Z at padded position (p, c) from the staged tile of g.  g is zero outside the image, so the tap loops run over the
// in-image rows / columns only; every in-image cell they read lies within h of a texel of this tile, so inside the box.
// taps = wx[0..K) then wy[0..K), in shared memory (dynamic indices).
template <int K>
__device__ __forceinline__ float zval_tile(const float* in_s, const float* taps, const PostParams& q, int gy0, int gx0, int p, int c) {
    constexpr int H = K / 2, BOXW = SwCfg<K>::BOXW;
    const int s0 = max(0, H - p), s1 = min(K, q.H + H - p), t0 = max(0, H - c), t1 = min(K, q.W + H - c);
    float acc = 0.f;
    for (int s = s0; s < s1; ++s) {
        const float* row = in_s + (p + s - H - gy0) * BOXW + (c - H - gx0);
        float hs = 0.f;
        for (int t = t0; t < t1; ++t) hs = fmaf(taps[t], row[t], hs);
        acc = fmaf(taps[K + s], hs, acc);
    }
    return acc;
}

// adds the fold terms (every preimage but the texel itself) to the Z the interior loop stored for this band texel
template <int K>
__device__ __forceinline__ void fold_texel(const float* in_s, const float* taps, const PostParams& q, int b, int gy0, int gx0, int y, int x) {
    float acc = 0.f;
#pragma unroll 1
    for (int u = 0; u < 3; ++u)
#pragma unroll 1
        for (int v = 0; v < 3; ++v) {
            int p, c;
            if ((u | v) != 0 && fold_preimage(u, y, q.H, K / 2, p) && fold_preimage(v, x, q.W, K / 2, c))
                acc += zval_tile<K>(in_s, taps, q, gy0, gx0, p, c);
        }
    q.out[((size_t)b * q.H + y) * q.W + x] += acc;
}

// Production form (kx == ky in {3, 5, 11}, W % 4 == 0, sides >= 16, 16-byte aligned g_out / g_in): the sliding-window
// kernel's skeleton.  One TMA load stages the tile of g + halo; the tensor map's out-of-bounds fill IS the zero extension
// of g, so the interior loop is the forward's without its reflect patch and writes Z.  Tiles that hold band texels then
// add the fold terms to those, read from the same staged tile (a few rows or columns of taps each: only the in-image part
// of a padded position's support is nonzero).  The register bound keeps ptxas from spilling
// (K = 11, two CTAs per SM: what its shared memory allows anyway) or from spending 94 registers (K = 5).
template <int K>
__global__ void __launch_bounds__(THREADS, K == 11 ? 2 : 4) blur_bwd_sw_kernel(const __grid_constant__ CUtensorMap tmap, const PostParams q) {
    typedef SwCfg<K> CF;
    constexpr int BOXW = CF::BOXW, BOXH = CF::BOXH, TH2 = CF::TH, RW = CF::RW, HK = CF::H;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* in_s = reinterpret_cast<float*>(smem_raw);                  // [BOXH][BOXW]
    __shared__ __align__(8) uint64_t bar;
    __shared__ float taps_s[2 * K];
    const int tiles_x = (q.W + SW_TW - 1) / SW_TW;
    const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x, b = blockIdx.y;
    const int x0 = tx * SW_TW, y0 = ty * TH2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    const int gx0 = x0 - CF::PADL, gy0 = y0 - HK;
    if (tid < 2 * K) taps_s[tid] = tid < K ? q.wx[tid] : q.wy[tid - K];
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(&bar, (uint32_t)(BOXW * BOXH * sizeof(float)));
        tma_load_3d(in_s, &tmap, &bar, gx0, gy0, b);
    }
    mbar_wait(&bar, 0);

    float wx[K], wy[K];
#pragma unroll
    for (int t = 0; t < K; ++t) { wx[t] = q.wx[t]; wy[t] = q.wy[t]; }
    const int x = x0 + 4 * lane;
    const float* colp = in_s + 4 * lane;
    float win[K][4];
#pragma unroll
    for (int rr = 0; rr < RW + K - 1; ++rr) {
        const float* rowp = colp + (warp * RW + rr) * BOXW;
        float v[4 * (1 + 2 * CF::NQ)];
#pragma unroll
        for (int w4 = 0; w4 < 1 + 2 * CF::NQ; ++w4) {
            const float4 a = *reinterpret_cast<const float4*>(rowp + 4 * w4);
            v[4 * w4] = a.x; v[4 * w4 + 1] = a.y; v[4 * w4 + 2] = a.z; v[4 * w4 + 3] = a.w;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float acc = 0.f;
#pragma unroll
            for (int t = 0; t < K; ++t) acc = fmaf(wx[t], v[CF::PADL - HK + j + t], acc);
            win[rr % K][j] = acc;
        }
        if (rr >= K - 1) {
            const int y = y0 + warp * RW + rr - (K - 1);
            float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int t = 0; t < K; ++t)
#pragma unroll
                for (int j = 0; j < 4; ++j) o[j] = fmaf(wy[t], win[(rr - (K - 1) + t) % K][j], o[j]);
            if (y < q.H && x < q.W)
                *reinterpret_cast<float4*>(q.out + ((size_t)b * q.H + y) * q.W + x) = make_float4(o[0], o[1], o[2], o[3]);
        }
    }

    // ---- fold epilogue: band texels of this tile (rows 1..h and H-1-h..H-2, the same for columns) ----
    const int ye = min(y0 + TH2, q.H), xe = min(x0 + SW_TW, q.W);
    const bool rows_hit = y0 <= HK || ye > q.H - 1 - HK, cols_hit = x0 <= HK || xe > q.W - 1 - HK;
    if (!rows_hit && !cols_hit) return;
    __syncthreads();                          // the band texels' Z values are written: the additions below read them
    // row band within the tile: [ra0, ra1) and [rb0, rb1), disjoint
    const int ra0 = max(y0, 1), ra1 = max(ra0, min(ye, HK + 1));
    const int rb0 = max(max(y0, q.H - 1 - HK), ra1), rb1 = max(rb0, min(ye, q.H - 1));
    const int nra = ra1 - ra0, nr = nra + (rb1 - rb0), ncols = xe - x0;
    for (int i = tid; i < nr * ncols; i += THREADS) {
        const int r = i / ncols, y = r < nra ? ra0 + r : rb0 + r - nra;
        fold_texel<K>(in_s, taps_s, q, b, gy0, gx0, y, x0 + i - r * ncols);
    }
    // column band within the tile, rows outside the row band
    const int ca0 = max(x0, 1), ca1 = max(ca0, min(xe, HK + 1));
    const int cb0 = max(max(x0, q.W - 1 - HK), ca1), cb1 = max(cb0, min(xe, q.W - 1));
    const int nca = ca1 - ca0, nc = nca + (cb1 - cb0), nrows = ye - y0;
    for (int i = tid; i < nrows * nc; i += THREADS) {
        const int r = i / nc, k = i - r * nc, y = y0 + r;
        if (in_fold_band(y, q.H, HK)) continue;
        fold_texel<K>(in_s, taps_s, q, b, gy0, gx0, y, k < nca ? ca0 + k : cb0 + k - nca);
    }
}

// no blur stage configured: pure streaming copy / noise / clip
__global__ void __launch_bounds__(THREADS) pointwise_kernel(const PostParams q) {
    // one item = a 4-texel quad of a row pair (rows 2 rp, 2 rp + 1): both loads in flight, one Philox call for the 8 variates
    const size_t quads_per_row = (size_t)(q.W + 3) / 4, pairs = (size_t)(q.H + 1) / 2;
    const size_t total = quads_per_row * pairs * q.B;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const bool vec = (q.W & 3) == 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int b = (int)(i / (quads_per_row * pairs));
        const size_t rem = i - (size_t)b * quads_per_row * pairs;
        const int rp = (int)(rem / quads_per_row), x0 = (int)(rem - (size_t)rp * quads_per_row) * 4;
        float v[2][4];
        bool live[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int y = 2 * rp + u;
            live[u] = y < q.H;
            const float* s = q.img + ((size_t)b * q.H + (live[u] ? y : 0)) * q.W + x0;
            if (vec) {
                const float4 a = __ldg(reinterpret_cast<const float4*>(s));
                v[u][0] = a.x; v[u][1] = a.y; v[u][2] = a.z; v[u][3] = a.w;
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) v[u][k] = x0 + k < q.W ? __ldg(s + k) : 0.f;
            }
        }
        const bool do_noise = q.noise && (q.gates ? q.gates[b * 2 + 1] != 0 : true);
        float za[4] = {0.f, 0.f, 0.f, 0.f}, zb[4] = {0.f, 0.f, 0.f, 0.f};
        if (do_noise && !q.noise_inj) normal8(q.seed, q.frame0 + (uint64_t)b, quadpair_index(q, 2 * rp, x0), za, zb);
        if (live[0]) {
            if (do_noise) noise_clip4z(q, b, 2 * rp, x0, v[0], za);
            store4(q, b, 2 * rp, x0, v[0]);
        }
        if (live[1]) {
            if (do_noise) noise_clip4z(q, b, 2 * rp + 1, x0, v[1], zb);
            store4(q, b, 2 * rp + 1, x0, v[1]);
        }
    }
}

// kornia 0.7.1 get_gaussian_kernel1d: x = i - k//2 (+0.5 for even k); exp(-x^2/(2 sigma^2)); normalised.
// Evaluated in fp32 like torch does (exp, then division by the fp32 sum).
static void gaussian_taps(int k, float sigma, float* w) {
    float sum = 0.f;
    for (int i = 0; i < k; ++i) {
        float x = (float)(i - k / 2);
        if (k % 2 == 0) x += 0.5f;
        w[i] = expf(-(x * x) / (2.0f * sigma * sigma));
        sum += w[i];
    }
    for (int i = 0; i < k; ++i) w[i] /= sum;
}

using tma::EncodeTiledFn;
using tma::get_encode;

// ---- silhouette (SURVEY.md 8(f) row 4) -------------------------------------------------------------------------------
// ApplySilhouette.post_process (fireflies/postprocessing/apply_silhouette.py:17-40): a filled disc of ones per frame,
// blurred 11x11 / sigma 5, multiplied into the image.  The disc is written analytically ((x-cx)^2 + (y-cy)^2 <= r^2; the
// reference rasterises it with cv2.circle, which is absent here: parity with OpenCV's circle is unpinned), the blur is the
// sliding-window kernel above and the product is its epilogue (PostParams::mul).
__global__ void __launch_bounds__(256) disc_mask_kernel(const int* __restrict__ discs, int B, int H, int W, float* __restrict__ mask) {
    const int b = blockIdx.y;
    const int cx = discs[3 * b], cy = discs[3 * b + 1], r = discs[3 * b + 2];
    const long long n4 = (long long)H * ((W + 3) / 4);
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n4; t += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(t / ((W + 3) / 4)), x0 = (int)(t % ((W + 3) / 4)) * 4;
        const long long dy2 = (long long)(y - cy) * (y - cy), r2 = (long long)r * r;
        float v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = ((long long)(x0 + k - cx) * (x0 + k - cx) + dy2 <= r2) ? 1.f : 0.f;
        float* o = mask + ((size_t)b * H + y) * W + x0;
        if (x0 + 4 <= W && (W & 3) == 0) *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
        else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (x0 + k < W) o[k] = v[k];
        }
    }
}

// ---- Perlin material textures (SURVEY.md 8(f) row 4) ---------------------------------------------------------------
// rand_perlin_2d_octaves (fireflies/sampling/noise_texture_lerp.py:8-62) with the lattice angles supplied by the caller
// (the reference draws them with torch.rand on the CPU generator; the Python mirror does the same, so the stream is
// consumed identically), then NoiseTextureLerpSampler.sample_train's min/max normalisation and colour lerp (:86-98).
__device__ __forceinline__ float torch_lerp(float a, float b, float w) {     // ATen lerp: two-sided form
    const float d = b - a;
    return w < 0.5f ? __fadd_rn(a, __fmul_rn(w, d)) : __fadd_rn(b, -__fmul_rn(d, __fadd_rn(1.f, -w)));
}
__device__ __forceinline__ float fade5(float t) {                             // 6 t^5 - 15 t^4 + 10 t^3, term by term like the lambda
    const float t3 = __fmul_rn(__fmul_rn(t, t), t), t4 = powf(t, 4.f), t5 = powf(t, 5.f);
    return __fadd_rn(__fadd_rn(__fmul_rn(6.f, t5), -__fmul_rn(15.f, t4)), __fmul_rn(10.f, t3));
}
// order-preserving float <-> int for atomicMin / atomicMax
__device__ __forceinline__ int f2ord(float f) { const int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7fffffff; }
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

struct PerlinParams {
    const float* angles;       // per octave (R0+1) x (R1+1) uniforms in [0,1), concatenated
    int H, W, res0, res1, octaves;
    float amp[8];              // float32(persistence^k)
    float* noise;              // [H, W]
    int* minmax;               // [2] ordered-int min / max
};

__global__ void __launch_bounds__(256) perlin_kernel(PerlinParams q) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = t < (long long)q.H * q.W;
    float acc = 0.f;
    if (live) {
        const int i = (int)(t / q.W), j = (int)(t - (long long)i * q.W);
        const float* ang = q.angles;
        int f = 1;
        for (int o = 0; o < q.octaves; ++o, f *= 2) {
            const int R0 = f * q.res0, R1 = f * q.res1;
            const int d0 = q.H / R0, d1 = q.W / R1;
            // torch.arange(0, R, R / shape) is start + i * step in double, stored as float32; then % 1
            const float a0 = (float)((double)i * ((double)R0 / (double)q.H)), a1 = (float)((double)j * ((double)R1 / (double)q.W));
            const float gx = a0 - floorf(a0), gy = a1 - floorf(a1);
            const int ci = i / d0, cj = j / d1;
            const float TWO_PI = 6.283185307179586f;
            float n[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int di = k & 1, dj = k >> 1;                   // n00, n10, n01, n11
                const float th = __fmul_rn(TWO_PI, __ldg(ang + (size_t)(ci + di) * (R1 + 1) + cj + dj));
                float sn, cs;
                sincosf(th, &sn, &cs);
                n[k] = __fadd_rn(__fmul_rn(gx - (float)di, cs), __fmul_rn(gy - (float)dj, sn));
            }
            const float t0 = fade5(gx), t1 = fade5(gy);
            const float v = __fmul_rn(1.4142135623730951f, torch_lerp(torch_lerp(n[0], n[1], t0), torch_lerp(n[2], n[3], t0), t1));
            acc = __fadd_rn(acc, __fmul_rn(q.amp[o], v));
            ang += (size_t)(R0 + 1) * (R1 + 1);
        }
        q.noise[t] = acc;
    }
    float mn = live ? acc : INFINITY, mx = live ? acc : -INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(q.minmax, f2ord(mn));
        atomicMax(q.minmax + 1, f2ord(mx));
    }
}

// out[c, i, j] = lerp(color_a[c], color_b[c], (noise - min) / (max - min))
__global__ void __launch_bounds__(256) noise_lerp_kernel(const float* __restrict__ noise, const int* __restrict__ minmax, long long n,
                                                         const float* __restrict__ ca, const float* __restrict__ cb, float* __restrict__ out) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const float mn = ord2f(minmax[0]), mx = ord2f(minmax[1]);
    const float w = __fdiv_rn(noise[t] - mn, mx - mn);
#pragma unroll
    for (int c = 0; c < 3; ++c) out[(size_t)c * n + t] = torch_lerp(__ldg(ca + c), __ldg(cb + c), w);
}

}  // namespace post
}  // namespace ffb

using namespace ffb;
using namespace ffb::post;

extern "C" int ffb_perlin_texture(const float* angles, int32_t H, int32_t W, int32_t res0, int32_t res1, int32_t octaves,
                                  double persistence, const float* color_a, const float* color_b, float* noise_scratch,
                                  int32_t* minmax_scratch, float* out, void* stream) {
    if (!angles || !noise_scratch || !minmax_scratch || H <= 0 || W <= 0 || res0 <= 0 || res1 <= 0)
        return fail_arg(FFB_E_ARG, "perlin_texture: bad argument");
    if (octaves < 1 || octaves > 8) return fail_arg(FFB_E_LIMIT, "perlin_texture: 1..8 octaves");
    if (out && (!color_a || !color_b)) return fail_arg(FFB_E_ARG, "perlin_texture: colours required with an output");
    const int top = 1 << (octaves - 1);
    if (H % (res0 * top) != 0 || W % (res1 * top) != 0)
        return fail_arg(FFB_E_ARG, "perlin_texture: shape must be a multiple of res * 2^(octaves-1) (as in the reference, whose tiling fails otherwise)");
    PerlinParams q;
    q.angles = angles; q.H = H; q.W = W; q.res0 = res0; q.res1 = res1; q.octaves = octaves;
    double a = 1.0;
    for (int o = 0; o < 8; ++o) { q.amp[o] = (float)a; a *= persistence; }
    q.noise = noise_scratch; q.minmax = minmax_scratch;
    cudaStream_t st = as_stream(stream);
    const int init[2] = {0x7f800000, (int)0x807fffff};       // ordered(+inf), ordered(-inf)
    FFB_CUDA(cudaMemcpyAsync(minmax_scratch, init, sizeof(init), cudaMemcpyHostToDevice, st));
    const long long n = (long long)H * W;
    perlin_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(q);
    FFB_CUDA(cudaGetLastError());
    if (out) {
        noise_lerp_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(noise_scratch, minmax_scratch, n, color_a, color_b, out);
        FFB_CUDA(cudaGetLastError());
    }
    return 0;
}

static int postprocess_impl(const ffb_post_desc* d, const float* img, const uint8_t* gates, const double* noise_injected,
                            const float* mul, float* out, void* stream);

extern "C" int ffb_postprocess(const ffb_post_desc* d, const float* img, const uint8_t* gates,
                               const double* noise_injected, float* out, void* stream) {
    return postprocess_impl(d, img, gates, noise_injected, nullptr, out, stream);
}

extern "C" int ffb_silhouette(const float* img, const int32_t* discs, int32_t B, int32_t H, int32_t W, float* mask_scratch, float* out,
                              void* stream) {
    if (!img || !discs || !mask_scratch || !out || B <= 0 || H <= 0 || W <= 0) return fail_arg(FFB_E_ARG, "silhouette: bad argument");
    if (B > 65535) return fail_arg(FFB_E_LIMIT, "silhouette: B > 65535");
    if (mask_scratch == out || mask_scratch == img) return fail_arg(FFB_E_ARG, "silhouette: the mask scratch must not alias the frames");
    cudaStream_t st = as_stream(stream);
    const long long n4 = (long long)H * ((W + 3) / 4);
    unsigned gx = (unsigned)((n4 + 255) / 256);
    if (gx > (unsigned)kNumSMs * 8) gx = (unsigned)kNumSMs * 8;
    disc_mask_kernel<<<dim3(gx, B), 256, 0, st>>>(discs, B, H, W, mask_scratch);
    FFB_CUDA(cudaGetLastError());
    ffb_post_desc d;
    memset(&d, 0, sizeof(d));
    d.B = B; d.H = H; d.W = W;
    d.blur_ky = 11; d.blur_kx = 11; d.blur_sy = 5.f; d.blur_sx = 5.f;      // apply_silhouette.py:31-35
    return postprocess_impl(&d, mask_scratch, nullptr, nullptr, img, out, stream);
}

static int postprocess_impl(const ffb_post_desc* d, const float* img, const uint8_t* gates, const double* noise_injected,
                            const float* mul, float* out, void* stream) {
    if (!d || !img || !out) return fail_arg(FFB_E_ARG, "postprocess: null pointer");
    if (d->B <= 0 || d->H <= 0 || d->W <= 0) return fail_arg(FFB_E_ARG, "postprocess: B, H, W must be positive");
    if (d->B > 65535) return fail_arg(FFB_E_LIMIT, "postprocess: B > 65535");
    const bool blur = d->blur_ky > 0 && d->blur_kx > 0;
    PostParams q;
    memset(&q, 0, sizeof(q));
    q.B = d->B; q.H = d->H; q.W = d->W;
    q.noise = d->noise; q.mean = d->noise_mean; q.stdv = d->noise_std; q.seed = d->seed; q.frame0 = d->frame0;
    q.img = img; q.gates = gates; q.noise_inj = noise_injected; q.mul = mul; q.out = out;
    cudaStream_t st = as_stream(stream);
    if (!blur) {
        const size_t total = (size_t)((d->W + 3) / 4) * ((d->H + 1) / 2) * d->B;
        size_t blocks = (total + THREADS - 1) / THREADS;
        if (blocks > (size_t)kNumSMs * 16) blocks = (size_t)kNumSMs * 16;
        pointwise_kernel<<<(unsigned)blocks, THREADS, 0, st>>>(q);
        FFB_CUDA(cudaGetLastError());
        return 0;
    }
    if (img == out) return fail_arg(FFB_E_ARG, "postprocess: img and out must not alias when blurring");
    if (d->blur_kx > KMAX || d->blur_ky > KMAX) return fail_arg(FFB_E_LIMIT, "postprocess: blur kernel size > 15");
    if (d->blur_kx % 2 == 0 || d->blur_ky % 2 == 0) return fail_arg(FFB_E_ARG, "postprocess: blur kernel sizes must be odd (all reference call sites are)");
    if (!(d->blur_sx > 0.f) || !(d->blur_sy > 0.f)) return fail_arg(FFB_E_ARG, "postprocess: blur sigma must be > 0");
    q.kx = d->blur_kx; q.ky = d->blur_ky; q.hx = q.kx / 2; q.hy = q.ky / 2;
    // torch reflect padding needs pad < dim
    if (q.hx >= d->W || q.hy >= d->H) return fail_arg(FFB_E_ARG, "postprocess: reflect border needs kernel/2 < image side");
    gaussian_taps(q.kx, d->blur_sx, q.wx);
    gaussian_taps(q.ky, d->blur_sy, q.wy);
    q.padl = (q.hx + 3) & ~3;
    q.boxw = (TW + q.padl + (q.kx - 1 - q.hx) + 3) & ~3;
    q.boxh = TH + q.ky - 1;
    const size_t smem = (size_t)q.boxh * (q.boxw + TW) * sizeof(float);
    const unsigned tiles = (unsigned)(((d->W + TW - 1) / TW) * ((d->H + TH - 1) / TH));
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    bool use_tma = (d->W % 4 == 0) && ((reinterpret_cast<uintptr_t>(img) & 15) == 0);
    if (use_tma) {
        EncodeTiledFn enc = get_encode();
        if (!enc) use_tma = false;
        else {
            cuuint64_t gdim[3] = {(cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->B};
            cuuint64_t gstr[2] = {(cuuint64_t)d->W * 4, (cuuint64_t)d->W * d->H * 4};
            cuuint32_t box[3] = {(cuuint32_t)q.boxw, (cuuint32_t)q.boxh, 1};
            cuuint32_t estr[3] = {1, 1, 1};
            CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(img), gdim, gstr, box, estr,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) use_tma = false;
        }
    }
    if (use_tma && q.kx == q.ky && (q.kx == 3 || q.kx == 5 || q.kx == 11) && d->W >= 16 && d->H >= 16) {
        // production path: sliding-window kernel; its TMA box differs from the generic kernel's
        CUtensorMap tm2;
        memset(&tm2, 0, sizeof(tm2));
        const int padl = (q.hx + 3) & ~3, rw = q.kx <= 5 ? 8 : 16;
        cuuint64_t gdim[3] = {(cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->B};
        cuuint64_t gstr[2] = {(cuuint64_t)d->W * 4, (cuuint64_t)d->W * d->H * 4};
        cuuint32_t box[3] = {(cuuint32_t)(SW_TW + 2 * padl), (cuuint32_t)(8 * rw + q.ky - 1), 1};
        cuuint32_t estr[3] = {1, 1, 1};
        if (get_encode()(&tm2, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(img), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS) {
            if (q.kx == 3) return launch_blur_sw<3, 3>(tm2, q, st);
            if (q.kx == 5) return launch_blur_sw<5, 5>(tm2, q, st);
            return launch_blur_sw<11, 11>(tm2, q, st);
        }
    }
    if (use_tma) {
        if (smem > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(blur_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        blur_kernel<true><<<dim3(tiles, d->B), THREADS, smem, st>>>(tmap, q);
    } else {
        if (smem > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(blur_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        blur_kernel<false><<<dim3(tiles, d->B), THREADS, smem, st>>>(tmap, q);
    }
    FFB_CUDA(cudaGetLastError());
    return 0;
}

template <int K>
static int launch_blur_bwd_sw(const PostParams& q, cudaStream_t st, bool* launched) {
    typedef SwCfg<K> CF;
    *launched = false;
    CUtensorMap tm;
    memset(&tm, 0, sizeof(tm));
    cuuint64_t gdim[3] = {(cuuint64_t)q.W, (cuuint64_t)q.H, (cuuint64_t)q.B};
    cuuint64_t gstr[2] = {(cuuint64_t)q.W * 4, (cuuint64_t)q.W * q.H * 4};
    cuuint32_t box[3] = {(cuuint32_t)CF::BOXW, (cuuint32_t)CF::BOXH, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    EncodeTiledFn enc = get_encode();
    if (!enc || enc(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(q.img), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return 0;
    const size_t smem = (size_t)CF::BOXW * CF::BOXH * sizeof(float);
    const unsigned tiles = (unsigned)(((q.W + SW_TW - 1) / SW_TW) * ((q.H + CF::TH - 1) / CF::TH));
    if (smem > 48 * 1024) FFB_CUDA(cudaFuncSetAttribute(blur_bwd_sw_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    blur_bwd_sw_kernel<K><<<dim3(tiles, q.B), THREADS, smem, st>>>(tm, q);
    FFB_CUDA(cudaGetLastError());
    *launched = true;
    return 0;
}

extern "C" int ffb_blur_bwd(const ffb_post_desc* d, const float* g_out, float* g_in, void* stream) {
    if (!d || !g_out || !g_in) return fail_arg(FFB_E_ARG, "blur_bwd: null pointer");
    if (d->B <= 0 || d->H <= 0 || d->W <= 0) return fail_arg(FFB_E_ARG, "blur_bwd: B, H, W must be positive");
    if (d->B > 65535) return fail_arg(FFB_E_LIMIT, "blur_bwd: B > 65535");
    if (d->noise != 0) return fail_arg(FFB_E_ARG, "blur_bwd: the noise stage has no backward (noise must be 0)");
    if (d->blur_ky <= 0 || d->blur_kx <= 0) return fail_arg(FFB_E_ARG, "blur_bwd: the descriptor has no blur stage");
    if (d->blur_kx > KMAX || d->blur_ky > KMAX) return fail_arg(FFB_E_LIMIT, "blur_bwd: blur kernel size > 15");
    if (d->blur_kx % 2 == 0 || d->blur_ky % 2 == 0) return fail_arg(FFB_E_ARG, "blur_bwd: blur kernel sizes must be odd");
    if (!(d->blur_sx > 0.f) || !(d->blur_sy > 0.f)) return fail_arg(FFB_E_ARG, "blur_bwd: blur sigma must be > 0");
    if (d->blur_kx / 2 >= d->W || d->blur_ky / 2 >= d->H) return fail_arg(FFB_E_ARG, "blur_bwd: reflect border needs kernel/2 < image side");
    const size_t bytes = (size_t)d->B * d->H * d->W * sizeof(float);
    const uintptr_t a = reinterpret_cast<uintptr_t>(g_out), c = reinterpret_cast<uintptr_t>(g_in);
    if (a < c + bytes && c < a + bytes) return fail_arg(FFB_E_ARG, "blur_bwd: g_out and g_in must not alias");
    PostParams q;
    memset(&q, 0, sizeof(q));
    q.B = d->B; q.H = d->H; q.W = d->W;
    q.kx = d->blur_kx; q.ky = d->blur_ky; q.hx = q.kx / 2; q.hy = q.ky / 2;
    gaussian_taps(q.kx, d->blur_sx, q.wx);
    gaussian_taps(q.ky, d->blur_sy, q.wy);
    q.img = g_out; q.out = g_in;
    cudaStream_t st = as_stream(stream);
    // the forward's sliding-window conditions, plus an aligned g_in for the 128-bit stores
    if (q.kx == q.ky && (q.kx == 3 || q.kx == 5 || q.kx == 11) && d->W % 4 == 0 && d->W >= 16 && d->H >= 16 && (a & 15) == 0 && (c & 15) == 0) {
        bool launched = false;
        int rc = q.kx == 3 ? launch_blur_bwd_sw<3>(q, st, &launched) : q.kx == 5 ? launch_blur_bwd_sw<5>(q, st, &launched)
                                                                                 : launch_blur_bwd_sw<11>(q, st, &launched);
        if (rc || launched) return rc;
    }
    const size_t total = bytes / sizeof(float);
    size_t blocks = (total + THREADS - 1) / THREADS;
    if (blocks > (size_t)kNumSMs * 16) blocks = (size_t)kNumSMs * 16;
    blur_bwd_kernel<<<(unsigned)blocks, THREADS, 0, st>>>(q);
    FFB_CUDA(cudaGetLastError());
    return 0;
}
